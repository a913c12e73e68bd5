// kidmp_api.cu - the C ABI of include/kidmp.h over the CUDA kernels.
// One translation unit: kidmp_tables.cuh (K3 table build) + kidmp_column.cuh / kidmp_cells.cuh (the step).
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -fmad=false (see kid_b200/build.py).
#include <cuda_runtime.h>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <cstdarg>
#include <cstdint>
#include <string>
#include <vector>
#include <map>
#include <mutex>
#include "kidmp_internal.h"
#include "kidmp_hostinit.h"
#include "kidmp_tables.cuh"
#include "kidmp_column.cuh"
#include "kidmp_cells.cuh"
#include "kidmp_kid.cuh"
#include "kidmp_wrf.cuh"

using namespace kidmp;

// kernel groups of one launch, in launch order (kidmp_kernel_names / kidmp_last_kernel_ms)
enum { KT_CLASSIFY = 0, KT_LISTS, KT_N0, KT_WARM, KT_ICE, KT_MIXNR, KT_FULL, KT_CARRIES, KT_SUBSTEPS, KT_FINISH, KT_DIAG, KT_N };

struct WorkSet {
  float* d_scratch = nullptr;                             // [nz*cols][SC_REC] hand-off records of the busy cells
  unsigned char* d_cls = nullptr;                         // [nz][cols] class byte of every cell
  int* d_colflag = nullptr;                               // [cols]
  int* d_work = nullptr;                                  // [count | list | mask | offset] of the cloudy columns
  unsigned* d_cells = nullptr;                            // [nz*cols] busy cells, class after class
  int* d_cellmeta = nullptr;                              // [192 | groups*64] class / key totals and starts, per-group bases
  unsigned* d_cellidx = nullptr;                          // [nz*cols] record number of every busy cell
  float* d_n0a = nullptr;                                 // [nz*cols] graupel intercept minima of S4
  float* d_ws = nullptr;                                  // [24][nz][cols] SoA workspace of the columns with sedimentation sub-steps
  double* d_coldiag = nullptr;                            // [2][cols] per-column water paths for the ordered domain sums
  int* d_colwork = nullptr;                               // [8 busy words | 8 colint | sub list | 2 colvmax][cols] of the column kernels
  long cols = 0; int nz = 0;
  cudaStream_t aux = nullptr;                             // second stream of a launch: k_n0_sweep, k_substeps
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  cudaEvent_t ev_lists_done = nullptr;                    // the work list is complete: k_n0_sweep may start
  cudaEvent_t ev_n0_done = nullptr;                       // k_n0_sweep is done: the cell kernels with graupel may start
};

struct kidmp_handle {
  int nsm = 148;
  kidmp_config cfg;
  std::string cache_path;
  int device = 0;
  cudaStream_t stream = nullptr, copy_in = nullptr, copy_out = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  KConst kc;
  HostBins hb;
  TableSet tabs{};
  char* d_tables = nullptr; size_t tables_bytes = 0;   // the slab behind tabs
  double* d_tnc_wev = nullptr;                          // table_dropEvap (M:4400-4439), made by the first aerosol-aware step
  float* d_aero = nullptr; size_t aero_floats = 0;      // staging of kidmp_mp_gt_driver_aero
  float table_ms = 0.f;
  bool tables_from_cache = false;
  long launches = 0;
  std::string err;
  // resident state
  long ncol = 0; int nz = 0;
  float* d_state = nullptr;      // [9][nz][ncol] fields, then p [nz][ncol]
  float* d_dz = nullptr;         // [nz]
  float* d_ppt = nullptr;        // [4][ncol]
  float* d_stage = nullptr;      // staging for layout conversion, [nz][ncol]
  double* d_partial = nullptr; long partial_chunks = 0;   // [chunks of one step][DIAG_BLOCKS][KIDMP_NDIAG] block sums of the domain diagnostics
  // Work buffers of one launch (a chunk of at most chunk_cols columns), sized for the worst case of the chunk
  WorkSet ws;
  // The launches of a step of up to 64 chunks are captured once in a CUDA graph and replayed while the arguments stay
  // the same ("graphs" option, KIDMP_GRAPHS; KIDMP_GRAPH_MAX: largest domain): a small domain is launch-bound (fifteen kernels of
  // a few microseconds: 0.297 -> 0.277 ms for one column), the 1 048 576-column step loses its launch gaps (3.45 -> 3.425 ms)
  int graphs = 1; long graph_max_cols = 1L << 24;
  struct StepGraph { cudaGraphExec_t exec = nullptr; StepArgs args{}; long key[7] = {}; long launches = 0; };
  StepGraph graph_cache[8]; int graph_next = 0;        // a few steps at a time: the three rotating buffers of kidmp_step's pipeline, resident state, a caller's arrays
  int simple = 1;                                         // "simple" option: columns without sub-steps skip k_carries (kidmp_cells.cuh)
  int classes = 1;                                        // "classes" option: 0 sends every busy cell to the general cell kernel (tests)
  // "timing" option: the kernels of a launch run one after the other on one stream with an event after each
  bool last_zero_copy = false;                            // the last kidmp_step wrote the changed columns straight into pinned host arrays
  int timing = 0; bool timing_valid = false;             // 1: kernels serialised on one stream; 2: the normal schedule, events on the main stream only
  cudaEvent_t ev_k[KT_N + 1] = {};
  long chunk_cols = 1048576;                              // columns per launch of the step kernels ("chunk" option, KIDMP_CHUNK)
  cudaEvent_t ev_done = nullptr;                          // end of the last step, on whatever stream it ran
  bool last_on_own_stream = true;
  double* d_diag = nullptr;
  float* d_rates = nullptr;                               // caller's device buffer (kidmp_set_rates_buffer) ...
  bool rates_on = false; float* d_rates_own = nullptr;    // ... or the handle's own, [36][nz][ncol] of the resident state (kidmp_enable_rates)
  float* d_kid = nullptr; size_t kid_floats = 0;   // staging of the KiD (k,i) arrays
  float* h_kid = nullptr; size_t h_kid_floats = 0; // pinned host twin of it
  float* d_pipe = nullptr; size_t pipe_floats = 0; int pipe_nz = 0; float* d_pipe_dz = nullptr;   // chunk pipeline of kidmp_step
  long pipe_chunk = 65536;
  float* h_ppt = nullptr; size_t h_ppt_floats = 0;       // pinned staging of ppt for the chunk pipeline
  cudaEvent_t pipe_ev[3][3] = {};
  float last_ms = 0.f;
  std::map<std::string, std::vector<double>> consts;   // named init constants for parity tests
  struct MultiCtx* multi = nullptr;                    // a handle over several devices (kidmp_config::ndev > 1): see "multi-device handle"
};

namespace {

std::string g_init_error;
std::mutex g_mu;

// Every entry point leaves the caller's current CUDA device as it found it (the host may be PyTorch or KiD's own code).
struct DevGuard {
  int prev = -1;
  explicit DevGuard(int d) { if (cudaGetDevice(&prev) != cudaSuccess) prev = -1; if (prev != d) cudaSetDevice(d); }
  ~DevGuard() { if (prev >= 0) cudaSetDevice(prev); }
};
struct DevRestore {                                    // for functions that walk over several devices
  int prev = -1;
  DevRestore() { if (cudaGetDevice(&prev) != cudaSuccess) prev = -1; }
  ~DevRestore() { if (prev >= 0) cudaSetDevice(prev); }
};

int fail(kidmp_handle* h, const char* fmt, ...) {
  char buf[512];
  va_list ap; va_start(ap, fmt); vsnprintf(buf, sizeof buf, fmt, ap); va_end(ap);
  if (h) h->err = buf; else g_init_error = buf;
  return 1;
}
#define CK(h, call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) return fail(h, "%s: %s", #call, cudaGetErrorString(e_)); } while (0)

template <class T> cudaError_t to_dev(const std::vector<T>& v, const T** out, std::vector<void*>& keep) {
  void* p = nullptr;
  cudaError_t e = cudaMalloc(&p, v.size() * sizeof(T));
  if (e != cudaSuccess) return e;
  keep.push_back(p);
  *out = (const T*)p;
  return cudaMemcpy(p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice);
}
template <class T> cudaError_t to_dev(const T* v, size_t n, const T** out, std::vector<void*>& keep) {
  return to_dev(std::vector<T>(v, v + n), out, keep);
}

uint64_t fnv(const void* p, size_t n, uint64_t h) {
  const unsigned char* c = (const unsigned char*)p;
  for (size_t i = 0; i < n; ++i) { h ^= c[i]; h *= 1099511628211ull; }
  return h;
}
// everything the table builders read: a cache written under other constants is refused
uint64_t table_key(const kidmp_handle* h) {
  uint64_t k = 1469598103934665603ull;
  k = fnv(&h->hb, sizeof h->hb, k);
  k = fnv(h->kc.cre, sizeof h->kc.cre, k); k = fnv(h->kc.crg, sizeof h->kc.crg, k);
  k = fnv(h->kc.cge, sizeof h->kc.cge, k); k = fnv(h->kc.cgg, sizeof h->kc.cgg, k);
  k = fnv(h->kc.cse, sizeof h->kc.cse, k); k = fnv(h->kc.cie, sizeof h->kc.cie, k);
  k = fnv(h->kc.ccg, sizeof h->kc.ccg, k);
  const int iw = h->kc.iiwarm; k = fnv(&iw, sizeof iw, k);
  return k ^ 0x6b69646d70743031ull;   // format tag "kidmpt01"
}
struct TabDesc { const void* base; long n; int stride; int member; bool f32; };
bool find_table(const kidmp_handle* h, const std::string& name, TabDesc& d) {
  static const char* g6[] = {"tcg_racg", "tmr_racg", "tcr_gacr", "tmg_gacr", "tnr_racg", "tnr_gacr"};
  static const char* s12[] = {"tcs_racs1", "tmr_racs1", "tcs_racs2", "tmr_racs2", "tcr_sacr1", "tms_sacr1",
                              "tcr_sacr2", "tms_sacr2", "tnr_racs1", "tnr_racs2", "tnr_sacr1", "tnr_sacr2"};
  static const char* f4[] = {"tpi_qrfz", "tpg_qrfz", "tni_qrfz", "tnr_qrfz"};
  static const char* c2[] = {"tpi_qcfz", "tni_qcfz"};
  static const char* i3[] = {"tps_iaus", "tni_iaus", "tpi_ide"};
  for (int q = 0; q < G_N; ++q) if (name == g6[q]) { d = {h->tabs.racg, N_RACG, G_N, q, false}; return true; }
  for (int q = 0; q < S_N; ++q) if (name == s12[q]) { d = {h->tabs.racs, N_RACS, S_N, q, false}; return true; }
  for (int q = 0; q < F_N; ++q) if (name == f4[q]) { d = {h->tabs.qrfz, N_QRFZ, F_N, q, false}; return true; }
  for (int q = 0; q < C_N; ++q) if (name == c2[q]) { d = {h->tabs.qcfz, N_QCFZ, C_N, q, false}; return true; }
  for (int q = 0; q < I_N; ++q) if (name == i3[q]) { d = {h->tabs.iaus, N_IAUS, I_N, q, false}; return true; }
  if (name == "t_Efrw") { d = {h->tabs.efrw, N_EF, 1, 0, true}; return true; }
  if (name == "t_Efsw") { d = {h->tabs.efsw, N_EF, 1, 0, true}; return true; }
  if (name == "tnc_wev" && h->d_tnc_wev) { d = {h->d_tnc_wev, (long)NBINS * NTB_C * NBINS, 1, 0, false}; return true; }   // (after the first aerosol-aware step)
  return false;
}

void publish_constants(kidmp_handle* h) {
  const KConst& k = h->kc;
  auto put = [&](const char* n, const float* a, int c) { h->consts[n] = std::vector<double>(a, a + c); };
  auto putd = [&](const char* n, const double* a, int c) { h->consts[n] = std::vector<double>(a, a + c); };
  put("cre", k.cre, 13); put("crg", k.crg, 13); put("cse", k.cse, 18); put("csg", k.csg, 18);
  put("cge", k.cge, 12); put("cgg", k.cgg, 12); put("cie", k.cie, 7); put("cig", k.cig, 7);
  for (int q = 0; q < 5; ++q) {
    put(("cce" + std::to_string(q + 1)).c_str(), k.cce[q], 15);
    put(("ccg" + std::to_string(q + 1)).c_str(), k.ccg[q], 15);
  }
  put("ocg1", k.ocg1, 15); put("ocg2", k.ocg2, 15);
  const float sc[] = {k.Nt_c, k.Sc3, k.D0i, k.xm0s, k.xm0g, k.rho_not, k.t1_qr_qc, k.t1_qr_qi, k.t2_qr_qi, k.t1_qg_qc,
                      k.t1_qs_qc, k.t1_qs_qi, k.t1_qr_ev, k.t2_qr_ev, k.t1_qs_sd, k.t2_qs_sd, k.t1_qg_sd, k.t2_qg_sd,
                      k.t1_qs_me, k.t2_qs_me, k.t1_qg_me, k.t2_qg_me, k.oig1, k.oig2, k.obmi, k.ore1, k.org1, k.org2,
                      k.org3, k.obmr, k.oams, k.obms, k.ocms, k.oge1, k.ogg1, k.ogg2, k.ogg3, k.oamg, k.obmg, k.ocmg,
                      k.am_r, k.am_g, k.am_i};
  put("scalars", sc, (int)(sizeof sc / sizeof sc[0]));
  const float of[] = {(float)k.nic1, (float)k.nic2, (float)k.nii2, (float)k.nii3, (float)k.nir2, (float)k.nir3,
                      (float)k.nis2, (float)k.nig2, (float)k.nig3, (float)k.niIN2};
  put("offsets", of, 10);
  const HostBins& b = h->hb;
  putd("Dc", b.Dc, NBINS); putd("Di", b.Di, NBINS); putd("Dr", b.Dr, NBINS); putd("Ds", b.Ds, NBINS); putd("Dg", b.Dg, NBINS);
  putd("t_Nc", b.t_Nc, NBINS); putd("dtc", b.dtc, NBINS); putd("dti", b.dti, NBINS); putd("dtr", b.dtr, NBINS);
  putd("dts", b.dts, NBINS); putd("dtg", b.dtg, NBINS);
}

struct TabAlloc { void** p; size_t bytes; };
std::vector<TabAlloc> table_allocs(kidmp_handle* h) {
  return {{(void**)&h->tabs.racg, (size_t)N_RACG * G_N * 8}, {(void**)&h->tabs.racs, (size_t)N_RACS * S_N * 8},
          {(void**)&h->tabs.qrfz, (size_t)N_QRFZ * F_N * 8}, {(void**)&h->tabs.qcfz, (size_t)N_QCFZ * C_N * 8},
          {(void**)&h->tabs.iaus, (size_t)N_IAUS * I_N * 8}, {(void**)&h->tabs.efrw, (size_t)N_EF * 4},
          {(void**)&h->tabs.efsw, (size_t)N_EF * 4}};
}

int load_cache(kidmp_handle* h) {   // 0 = loaded
  FILE* f = fopen(h->cache_path.c_str(), "rb");
  if (!f) return 1;
  uint64_t key = 0;
  bool ok = fread(&key, 8, 1, f) == 1 && key == table_key(h);
  std::vector<char> buf;
  for (auto& a : table_allocs(h)) {
    if (!ok) break;
    buf.resize(a.bytes);
    ok = fread(buf.data(), 1, a.bytes, f) == a.bytes &&
         cudaMemcpy(*a.p, buf.data(), a.bytes, cudaMemcpyHostToDevice) == cudaSuccess;
  }
  fclose(f);
  return ok ? 0 : 1;
}

int build_device_tables(kidmp_handle* h, const hostinit::Prep& pp) {
  std::vector<void*> keep;
  TablePrep tp{};
  TableScratch sc{};
  cudaError_t e = cudaSuccess;
  auto up = [&](cudaError_t r) { if (e == cudaSuccess) e = r; };
  up(to_dev(pp.lamr, &tp.lamr, keep)); up(to_dev(pp.N0_r, &tp.N0_r, keep));
  up(to_dev(pp.lamg, &tp.lamg, keep)); up(to_dev(pp.N0_g, &tp.N0_g, keep));
  up(to_dev(pp.s_Mrat, &tp.s_Mrat, keep)); up(to_dev(pp.s_M0, &tp.s_M0, keep));
  up(to_dev(pp.s_slam1, &tp.s_slam1, keep)); up(to_dev(pp.s_slam2, &tp.s_slam2, keep));
  up(to_dev(pp.lamc, &tp.lamc, keep)); up(to_dev(pp.N0_c, &tp.N0_c, keep));
  up(to_dev(pp.i_lami, &tp.i_lami, keep)); up(to_dev(pp.i_N0, &tp.i_N0, keep));
  up(to_dev(pp.i_tpi_ide, &tp.i_tpi_ide, keep)); up(to_dev(pp.i_branch, &tp.i_branch, keep));
  const HostBins& b = h->hb;
  up(to_dev(b.Dc, NBINS, &tp.Dc, keep)); up(to_dev(b.dtc, NBINS, &tp.dtc, keep));
  up(to_dev(b.Di, NBINS, &tp.Di, keep)); up(to_dev(b.dti, NBINS, &tp.dti, keep));
  up(to_dev(b.Dr, NBINS, &tp.Dr, keep)); up(to_dev(b.dtr, NBINS, &tp.dtr, keep));
  up(to_dev(b.Ds, NBINS, &tp.Ds, keep)); up(to_dev(b.dts, NBINS, &tp.dts, keep));
  up(to_dev(b.Dg, NBINS, &tp.Dg, keep)); up(to_dev(b.dtg, NBINS, &tp.dtg, keep));
  up(to_dev(b.r_r, NTB_R, &tp.r_r, keep)); up(to_dev(b.r_c, NTB_C, &tp.r_c, keep));
  up(to_dev(b.r_i, NTB_I, &tp.r_i, keep)); up(to_dev(b.Nt_i, NTB_I1, &tp.Nt_i, keep));
  tp.t_Nc1 = b.t_Nc[0]; tp.nu_c_fz = pp.nu_c_fz; tp.xm0g = h->kc.xm0g; tp.obmr = h->kc.obmr; tp.D0s = KP_D0S;
  tp.am_r = h->kc.am_r; tp.am_g = h->kc.am_g; tp.am_i = h->kc.am_i; tp.am_s = pp.am_s;
  memcpy(tp.Texp, pp.Texp, sizeof tp.Texp);
  const size_t nR = (size_t)NTB_R * NTB_R1 * NBINS, nG = (size_t)NTB_G * NTB_G1 * NBINS, nS = (size_t)NTB_T * NTB_S * NBINS;
  void* p = nullptr;
  up(cudaMalloc(&p, nR * 8)); keep.push_back(p); sc.N_r = (double*)p;
  up(cudaMalloc(&p, nG * 8)); keep.push_back(p); sc.N_g = (double*)p;
  up(cudaMalloc(&p, nS * 8)); keep.push_back(p); sc.N_s = (double*)p;
  if (e == cudaSuccess) e = build_tables_dev(tp, h->tabs, sc, !h->kc.iiwarm, h->stream, &h->table_ms, &h->launches);
  for (void* q : keep) cudaFree(q);
  if (e != cudaSuccess) return fail(h, "table build: %s", cudaGetErrorString(e));
  return 0;
}

// The scalars of thompson_init live in ONE __constant__ block per device (`ck`) and one __device__ double (the graupel
// intercept constant): the handle that ran last on a device owns them.  A change of owner is ordered on the device: the
// new owner's stream first waits for the previous owner's last step, then uploads on that same stream, so neither
// handle's kernels can see the other's constants.
constexpr int MAX_DEVICES = 64;
kidmp_handle* g_const_owner[MAX_DEVICES] = {};
int ensure_constants(kidmp_handle* h, cudaStream_t s) {
  std::lock_guard<std::mutex> lk(g_mu);
  kidmp_handle*& owner = g_const_owner[h->device];
  if (owner != h) {
    if (owner && owner->ev_done) CK(h, cudaStreamWaitEvent(s, owner->ev_done, 0));
    CK(h, cudaMemcpyToSymbolAsync(ck, &h->kc, sizeof(KConst), 0, cudaMemcpyHostToDevice, s));
    k_n0_lo<<<1, 1, 0, s>>>();                       // the per-run graupel intercept constant (kidmp_column.cuh)
    owner = h;
  }
  return 0;
}

void free_work(WorkSet& w) {
  void* old[] = {w.d_scratch, w.d_cls, w.d_colflag, w.d_work, w.d_cells, w.d_cellmeta, w.d_coldiag, w.d_colwork, w.d_cellidx, w.d_ws, w.d_n0a};
  for (void* q : old) if (q) cudaFree(q);
  w.d_scratch = nullptr; w.d_cls = nullptr; w.d_colflag = nullptr; w.d_work = nullptr; w.d_cells = nullptr;
  w.d_cellmeta = nullptr; w.d_coldiag = nullptr; w.d_colwork = nullptr; w.d_cellidx = nullptr; w.d_ws = nullptr; w.d_n0a = nullptr; w.cols = 0; w.nz = 0;
}
int ensure_work(kidmp_handle* h, long cols, int nz) {
  WorkSet& w = h->ws;
  if (cols <= w.cols && nz <= w.nz) return 0;
  const long C = cols > w.cols ? cols : w.cols;
  const int Z = nz > w.nz ? nz : w.nz;
  // Only this handle's steps use the buffers that go away, and each has ended at ev_done (the k_scatter_host that follows a
  // pipelined step is waited for before step_pipelined returns).  A device-wide wait would also fail another thread's capture.
  CK(h, cudaEventSynchronize(h->ev_done));
  free_work(w);
  const size_t cells = (size_t)C * Z;
  const long ngroups = (C + 31) / 32, lblocks = (C + LIST_TILE - 1) / LIST_TILE;
  CK(h, cudaMalloc((void**)&w.d_scratch, cells * SC_REC * 4));
  CK(h, cudaMalloc((void**)&w.d_cls, cells));
  CK(h, cudaMalloc((void**)&w.d_colflag, (size_t)C * 4));
  CK(h, cudaMalloc((void**)&w.d_work, (size_t)(C + 8 + 2 * ngroups) * 4));
  CK(h, cudaMalloc((void**)&w.d_cells, cells * 4));
  CK(h, cudaMalloc((void**)&w.d_cellidx, cells * 4));
  CK(h, cudaMalloc((void**)&w.d_ws, cells * WS_N * 4));
  CK(h, cudaMalloc((void**)&w.d_n0a, cells * 4));
  CK(h, cudaMalloc((void**)&w.d_cellmeta, (size_t)(192 + lblocks * (LIST_TILE / 32) * 64) * 4));
  CK(h, cudaMalloc((void**)&w.d_coldiag, (size_t)C * 2 * 8));
  CK(h, cudaMalloc((void**)&w.d_colwork, (size_t)C * 19 * 4));
  w.cols = C; w.nz = Z;
  return 0;
}

// launch shape of the cell kernels: threads per block, blocks per SM, stage barriers of the lockstep blocks (bit i =
// LOCKBAR(i) of kidmp_cells.cuh; 0 = warps run free).  Measured alternatives: profiles/r02_cells_variants.md
#ifndef KC_WARM_T
#define KC_WARM_T 256
#endif
#ifndef KC_WARM_B
#define KC_WARM_B 4
#endif
#ifndef KC_WARM_BARS
#define KC_WARM_BARS 11
#endif
#ifndef KC_ICE_T
#define KC_ICE_T 256
#endif
#ifndef KC_ICE_B
#define KC_ICE_B 4
#endif
#ifndef KC_ICE_BARS
#define KC_ICE_BARS 11
#endif
#ifndef KC_MIXNR_T
#define KC_MIXNR_T 256
#endif
#ifndef KC_MIXNR_B
#define KC_MIXNR_B 3
#endif
#ifndef KC_MIXNR_BARS
#define KC_MIXNR_BARS 11
#endif
#ifndef KC_FULL_T
#define KC_FULL_T 256
#endif
#ifndef KC_FULL_B
#define KC_FULL_B 3
#endif
#ifndef KC_FULL_BARS
#define KC_FULL_BARS 11
#endif

#ifndef KC_AERO_WARM_B
#define KC_AERO_WARM_B 3
#endif
#ifndef KC_AERO_ICE_B
#define KC_AERO_ICE_B 3
#endif
#ifndef KC_AERO_MIX_B
#define KC_AERO_MIX_B 2
#endif
template <bool RATES, bool AERO>
void launch_cells(kidmp_handle* h, const StepArgs& a, int nsm, cudaStream_t s, cudaEvent_t n0_done) {
  auto mark = [&](int q) { if (h->timing) cudaEventRecord(h->ev_k[q + 1], s); };
  // (the aerosol-aware instantiations carry more live values: one block per SM less keeps them out of local memory)
  constexpr int WB = AERO ? KC_AERO_WARM_B : KC_WARM_B, IB = AERO ? KC_AERO_ICE_B : KC_ICE_B, MB = AERO ? KC_AERO_MIX_B : KC_MIXNR_B,
                FB = AERO ? KC_AERO_MIX_B : KC_FULL_B;
  k_cells<KC_WARM, KC_WARM_T, WB, KC_WARM_BARS, RATES, AERO><<<nsm * WB, KC_WARM_T, 0, s>>>(a);
  mark(KT_WARM);
  k_cells<KC_ICE, KC_ICE_T, IB, KC_ICE_BARS, RATES, AERO><<<nsm * IB, KC_ICE_T, 0, s>>>(a);
  mark(KT_ICE);
  if (n0_done) cudaStreamWaitEvent(s, n0_done, 0);     // only the classes with graupel read the intercept minima of k_n0_sweep
  k_cells<KC_MIXNR, KC_MIXNR_T, MB, KC_MIXNR_BARS, RATES, AERO><<<nsm * MB, KC_MIXNR_T, 0, s>>>(a);
  mark(KT_MIXNR);
  k_cells<KC_FULL, KC_FULL_T, FB, KC_FULL_BARS, RATES, AERO><<<nsm * FB, KC_FULL_T, 0, s>>>(a);
  mark(KT_FULL);
}

// One step over [ncol] columns whose arrays have row stride ld, in launches of at most chunk_cols columns on the caller's
// stream (the work buffers are sized for one launch: 29 hand-off planes would otherwise grow with the domain).  Columns are
// independent, so the chunking changes no result.
int launch_step(kidmp_handle* h, const StepArgs& a0, cudaStream_t s) {
  if (a0.nz < 2 || a0.nz > 256) return fail(h, "nz=%d outside [2,256]", a0.nz);
  if (a0.ncol < 1) return fail(h, "ncol=%ld", a0.ncol);
  if (!(a0.dt > 0.f)) return fail(h, "dt must be positive");
  const long chunk = h->chunk_cols;
  const long cap = a0.ncol < chunk ? a0.ncol : chunk;
  const long nchunks = (a0.ncol + chunk - 1) / chunk;
  if (cap > (1L << 24)) return fail(h, "chunk of %ld columns: at most 16 777 216 per launch (set_option \"chunk\")", cap);
  if ((double)cap * a0.nz >= 4.0e9) return fail(h, "chunk of %ld columns x %d levels does not fit the 32-bit cell index", cap, a0.nz);
  if (ensure_work(h, cap, a0.nz)) return 1;
  // the work set is the handle's: a step on another stream than the last one starts after it
  CK(h, cudaStreamWaitEvent(s, h->ev_done, 0));
  if (ensure_constants(h, s)) return 1;
  if (h->partial_chunks < nchunks) {
    if (h->d_partial) { CK(h, cudaEventSynchronize(h->ev_done)); cudaFree(h->d_partial); h->d_partial = nullptr; h->partial_chunks = 0; }
    CK(h, cudaMalloc((void**)&h->d_partial, (size_t)nchunks * DIAG_BLOCKS * KIDMP_NDIAG * 8));
    h->partial_chunks = nchunks;
  }
  // Replay the captured graph of this very step (all its chunks), or capture it now.
  const bool graphable = h->graphs && !h->timing && nchunks <= 64 && a0.ncol <= h->graph_max_cols;
  // (a handle setting that a captured launch reads belongs in the key: a replay after the setting changed would run the old one)
  const long gkey[7] = {(long)(size_t)h->ws.d_scratch, h->ws.cols, (long)h->ws.nz, (long)h->simple, (long)(size_t)h->d_partial,
                        chunk, (long)h->classes};
  kidmp_handle::StepGraph* hit = nullptr;
  if (graphable)
    for (auto& g : h->graph_cache)
      if (g.exec && !memcmp(&g.args, &a0, sizeof a0) && !memcmp(g.key, gkey, sizeof gkey)) { hit = &g; break; }
  if (hit) {
    CK(h, cudaGraphLaunch(hit->exec, s));
    h->launches += hit->launches;
    h->timing_valid = false;
    CK(h, cudaEventRecord(h->ev_done, s));
    h->last_on_own_stream = (s == h->stream);
    return 0;
  }
  bool capturing = false;
  const long launches_before = h->launches;
  kidmp_handle::StepGraph& slot = h->graph_cache[h->graph_next];
  if (graphable) {
    h->graph_next = (h->graph_next + 1) % 8;
    if (slot.exec) { cudaEventSynchronize(h->ev_done); cudaGraphExecDestroy(slot.exec); slot.exec = nullptr; }   // (its last replay has ended)
    capturing = cudaStreamBeginCapture(s, cudaStreamCaptureModeRelaxed) == cudaSuccess;
    if (!capturing) cudaGetLastError();                 // (a stream that cannot be captured: plain launches)
  }
  struct CaptureGuard {                                 // an error path must not leave the stream in capture mode
    cudaStream_t s; bool* on;
    ~CaptureGuard() { if (*on) { cudaGraph_t g = nullptr; cudaStreamEndCapture(s, &g); if (g) cudaGraphDestroy(g); cudaGetLastError(); } }
  } capture_guard{s, &capturing};
  // the handle's own rate buffer starts every step at zero: clear-sky columns have no process at all
  if (a0.rates && a0.rates == h->d_rates_own) CK(h, cudaMemsetAsync(h->d_rates_own, 0, (size_t)KIDMP_NRATES * a0.nz * a0.ld * 4, s));
  const WorkSet& w = h->ws;
  long ci = 0;
  for (long c0 = 0; c0 < a0.ncol; c0 += chunk, ++ci) {
    StepArgs a = a0;
    a.ncol = (a0.ncol - c0 < chunk) ? (a0.ncol - c0) : chunk;
    for (int q = 0; q < KIDMP_NFIELDS; ++q) a.f[q] = a0.f[q] + c0;
    a.p = a0.p + c0; a.ppt = a0.ppt + c0;
    if (a0.dz_col) a.dz_col = a0.dz_col + c0;
    if (a0.rates) a.rates = a0.rates + c0;
    if (a0.nc) { a.nc = a0.nc + c0; a.nwfa = a0.nwfa + c0; a.nifa = a0.nifa + c0; a.w = a0.w + c0; }
    const long ngroups = (a.ncol + 31) / 32, lblocks = (a.ncol + LIST_TILE - 1) / LIST_TILE;
    a.scratch = w.d_scratch; a.scratch_b = w.d_scratch + (size_t)w.cols * w.nz * SC_HALF; a.cellidx = w.d_cellidx; a.cls = w.d_cls; a.colflag = w.d_colflag;
    a.work_count = w.d_work; a.work_list = w.d_work + 8;
    a.work_mask = (unsigned*)(w.d_work + 8 + a.ncol); a.work_offset = w.d_work + 8 + a.ncol + ngroups;
    a.cell_list = w.d_cells; a.cell_count = w.d_cellmeta; a.sub_count = w.d_cellmeta + 5; a.cell_kstart = w.d_cellmeta + 8;
    a.cell_hist = w.d_cellmeta + 64; a.cell_start = w.d_cellmeta + 128; a.cell_base = w.d_cellmeta + 192;
    a.busy = (unsigned*)w.d_colwork; a.colint = w.d_colwork + 8 * w.cols; a.sub_list = w.d_colwork + 16 * w.cols; a.colvmax = w.d_colwork + 17 * w.cols;
    a.ws = w.d_ws; a.ws_cols = w.cols; a.n0a = w.d_n0a;
    a.coldiag = w.d_coldiag; a.diag_partial = h->d_partial + (size_t)ci * DIAG_BLOCKS * KIDMP_NDIAG; a.nsm = h->nsm; a.no_simple = h->simple ? 0 : 1;
    a.no_classes = h->classes ? 0 : 1;
    // second stream of the launch; in timing mode everything runs on one stream, one kernel after the other
    const bool serial = h->timing == 1;
    cudaStream_t x = serial ? s : w.aux;
    auto mark = [&](int q) { if (h->timing) cudaEventRecord(h->ev_k[q + 1], s); };
    auto fork = [&](cudaEvent_t e, cudaStream_t from, cudaStream_t to) {
      if (from != to) { cudaEventRecord(e, from); cudaStreamWaitEvent(to, e, 0); }
    };
    CK(h, cudaMemsetAsync(w.d_cellmeta, 0, 128 * 4, s));
    if (h->timing) CK(h, cudaEventRecord(h->ev_k[0], s));
    k_classify<<<(unsigned)((a.ncol + 127) / 128), 128, 0, s>>>(a);
    CK(h, cudaMemsetAsync(a.colvmax, 0, (size_t)2 * w.cols * 4, s));
    mark(KT_CLASSIFY);
    // The classification left the key histogram of the busy cells: first entry of every key and class, the work list of
    // the cloudy columns, then the list of the busy cells.  Second stream: the graupel intercept sweep (needs the work list
    // only; the cell kernels with graupel wait for it).
    k_cell_offsets<<<1, 64, 0, s>>>(a);
    k_list_scan<<<1, 1024, 0, s>>>(a.work_mask, (int)ngroups, a.work_offset, a.work_count);
    k_list_fill<<<(unsigned)((ngroups * 32 + 255) / 256), 256, 0, s>>>(a.work_mask, a.work_offset, (int)ngroups, a.work_list);
    if (serial) {
      k_cell_fill<<<(unsigned)lblocks, LIST_TILE, 0, s>>>(a);
      mark(KT_LISTS);
      if (!h->kc.iiwarm) k_n0_sweep<<<(unsigned)((a.ncol + 127) / 128), 128, 0, s>>>(a);
      mark(KT_N0);
    } else {
      fork(w.ev_lists_done, s, x);                   // (recorded after k_list_fill)
      // the number of cloudy columns is only known on the device: grids for the worst case, surplus blocks leave at once
      if (!h->kc.iiwarm) k_n0_sweep<<<(unsigned)((a.ncol + 127) / 128), 128, 0, x>>>(a);
      k_cell_fill<<<(unsigned)lblocks, LIST_TILE, 0, s>>>(a);
      CK(h, cudaEventRecord(w.ev_n0_done, x));       // the sweep runs beside k_cell_fill and the warm and ice cell kernels
      mark(KT_LISTS); mark(KT_N0);
    }
    cudaEvent_t n0_done = serial ? nullptr : w.ev_n0_done;
    const bool aero = a.nc != nullptr;                  // (an aerosol-aware step has no process-rate buffer: checked by its entry point)
    if (aero) launch_cells<false, true>(h, a, h->nsm, s, n0_done);
    else if (a.rates) launch_cells<true, false>(h, a, h->nsm, s, n0_done);
    else launch_cells<false, false>(h, a, h->nsm, s, n0_done);
    k_carries<<<(unsigned)((a.ncol + 63) / 64), 64, 0, s>>>(a);
    mark(KT_CARRIES);
    // the columns with sedimentation sub-steps on the second stream, the others on this one: disjoint columns
    fork(w.ev_fork, s, x);
    const unsigned sgrid = (unsigned)(ngroups < h->nsm * 16 ? ngroups : h->nsm * 16);
    if (aero) k_substeps<false, true><<<sgrid, 32, 0, x>>>(a);
    else if (a.rates) k_substeps<true, false><<<sgrid, 32, 0, x>>>(a); else k_substeps<false, false><<<sgrid, 32, 0, x>>>(a);
    mark(KT_SUBSTEPS);
    if (aero) k_finish<false, true><<<(unsigned)ngroups, 32, 0, s>>>(a);
    else if (a.rates) k_finish<true, false><<<(unsigned)ngroups, 32, 0, s>>>(a); else k_finish<false, false><<<(unsigned)ngroups, 32, 0, s>>>(a);
    mark(KT_FINISH);
    fork(w.ev_join, x, s);
    k_diag_columns<<<DIAG_BLOCKS, 256, 0, s>>>(a, (a.ncol + DIAG_BLOCKS - 1) / DIAG_BLOCKS);
    h->launches += h->kc.iiwarm ? 13 : 14;
  }
  // the block sums of all launches, in column order
  k_diag_reduce<<<KIDMP_NDIAG, 256, 0, s>>>(h->d_partial, (int)(nchunks * DIAG_BLOCKS), h->d_diag);
  ++h->launches;
  if (h->timing) cudaEventRecord(h->ev_k[KT_DIAG + 1], s);
  h->timing_valid = h->timing != 0;
  if (capturing) {
    cudaGraph_t g = nullptr;
    capturing = false;                                  // (the guard has nothing left to end)
    CK(h, cudaStreamEndCapture(s, &g));
    const cudaError_t ie = cudaGraphInstantiate(&slot.exec, g, 0);
    cudaGraphDestroy(g);
    if (ie != cudaSuccess) { slot.exec = nullptr; return fail(h, "cudaGraphInstantiate: %s", cudaGetErrorString(ie)); }
    slot.args = a0; memcpy(slot.key, gkey, sizeof gkey);
    slot.launches = h->launches - launches_before;
    CK(h, cudaGraphLaunch(slot.exec, s));
  }
  CK(h, cudaGetLastError());
  CK(h, cudaEventRecord(h->ev_done, s));
  h->last_on_own_stream = (s == h->stream);
  return 0;
}

void free_state(kidmp_handle* h) {
  if (h->d_rates_own) cudaFree(h->d_rates_own);
  h->d_rates_own = nullptr;
  if (h->d_state) cudaFree(h->d_state);
  if (h->d_dz) cudaFree(h->d_dz);
  if (h->d_ppt) cudaFree(h->d_ppt);
  if (h->d_stage) cudaFree(h->d_stage);
  h->d_state = h->d_dz = h->d_ppt = h->d_stage = nullptr;
  h->ncol = 0; h->nz = 0;
}

inline float* field_ptr(kidmp_handle* h, int q) { return h->d_state + (size_t)q * h->nz * h->ncol; }

StepArgs resident_args(kidmp_handle* h, float dt) {
  StepArgs a{};
  a.ncol = h->ncol; a.ld = h->ncol; a.nz = h->nz; a.dt = dt;
  for (int q = 0; q < KIDMP_NFIELDS; ++q) a.f[q] = field_ptr(h, q);
  a.p = field_ptr(h, KIDMP_NFIELDS);
  a.dz = h->d_dz; a.ppt = h->d_ppt; a.rates = h->d_rates ? h->d_rates : h->d_rates_own;
  return a;
}

// host <-> device copy of one field with layout conversion
int put_field(kidmp_handle* h, int layout, const float* src, float* dst) {
  const size_t bytes = (size_t)h->ncol * h->nz * 4;
  if (layout == KIDMP_COL_FASTEST || h->ncol == 1) {
    CK(h, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, h->stream));
  } else {
    CK(h, cudaMemcpyAsync(h->d_stage, src, bytes, cudaMemcpyHostToDevice, h->stream));
    dim3 g((unsigned)((h->ncol + 31) / 32), (unsigned)((h->nz + 31) / 32)), b(32, 8);
    k_transpose<<<g, b, 0, h->stream>>>(h->d_stage, dst, h->ncol, h->nz, 1);
    ++h->launches;
  }
  return 0;
}
int get_field(kidmp_handle* h, int layout, const float* src, float* dst) {
  const size_t bytes = (size_t)h->ncol * h->nz * 4;
  if (layout == KIDMP_COL_FASTEST || h->ncol == 1) {
    CK(h, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, h->stream));
  } else {
    dim3 g((unsigned)((h->ncol + 31) / 32), (unsigned)((h->nz + 31) / 32)), b(32, 8);
    k_transpose<<<g, b, 0, h->stream>>>(src, h->d_stage, h->ncol, h->nz, 0);
    ++h->launches;
    CK(h, cudaMemcpyAsync(dst, h->d_stage, bytes, cudaMemcpyDeviceToHost, h->stream));
    CK(h, cudaStreamSynchronize(h->stream));   // d_stage is reused by the next field
  }
  return 0;
}


// ---- multi-device handle -------------------------------------------------------------------------------------------------
// kidmp_config::ndev > 1: one handle owns a full single-device handle per GPU (streams, tables, constants, work buffers) and
// a single-process NCCL communicator over them.  Columns are independent (I:54, M:1156-1177), so the host arrays are cut into
// contiguous column ranges, one per device, with no exchange on the data path; kidmp_diag returns the NCCL all-reduced domain
// sums (the device twin of the column means of I:255-275).  NCCL is loaded at run time (libnccl.so.2, or KIDMP_NCCL_LIB):
// a single-device handle needs no NCCL at all.
}  // namespace
#include <dlfcn.h>
#include <thread>
extern "C" {
static int step_pipelined(kidmp_handle* h, long ncol, int nz, float dt, float* const fields[KIDMP_NFIELDS], const float* p,
                          const float* dz, float* ppt, long hld);
}
struct MultiCtx {
  std::vector<kidmp_handle*> dev;
  void* lib = nullptr;
  std::vector<void*> comms;                          // ncclComm_t
  int (*CommInitAll)(void**, int, const int*) = nullptr;
  int (*CommDestroy)(void*) = nullptr;
  int (*AllReduce)(const void*, void*, size_t, int, int, void*, cudaStream_t) = nullptr;
  int (*GroupStart)() = nullptr;
  int (*GroupEnd)() = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
  std::vector<double*> d_red;                        // [8] per device: the sums being reduced
  long ncol = 0; int nz = 0;                         // resident state: columns of the whole domain
};
namespace {
void shard(long ncol, int d, int n, long& c0, long& c1) { c0 = ncol * d / n; c1 = ncol * (d + 1) / n; }

// run fn(d) for every device at the same time (the entry points block until their device is done); returns the first error
template <class F> int on_all(kidmp_handle* h, F fn) {
  DevRestore restore_;                                 // (fn(0) runs on the caller's thread)
  MultiCtx* m = h->multi;
  const int n = (int)m->dev.size();
  std::vector<int> rc(n, 0);
  std::vector<std::thread> th;
  for (int d = 1; d < n; ++d) th.emplace_back([&, d] { rc[d] = fn(d); });
  rc[0] = fn(0);
  for (auto& t : th) t.join();
  for (int d = 0; d < n; ++d) if (rc[d]) return fail(h, "device %d: %s", m->dev[d]->device, m->dev[d]->err.c_str());
  return 0;
}

int multi_step(kidmp_handle* h, long ncol, int nz, float dt, int layout, float* const fields[KIDMP_NFIELDS], const float* p,
               const float* dz, float* ppt) {
  MultiCtx* m = h->multi;
  const int n = (int)m->dev.size();
  for (int q = 0; q < KIDMP_NFIELDS; ++q) if (!fields[q]) return fail(h, "step: field %d is null", q);
  if (ncol < 1 || nz < 2 || nz > 256 || !(dt > 0.f)) return fail(h, "step: ncol=%ld nz=%d dt=%g", ncol, nz, (double)dt);
  return on_all(h, [&](int d) -> int {
    kidmp_handle* c = m->dev[d];
    long c0, c1;
    shard(ncol, d, n, c0, c1);
    if (c1 <= c0) return 0;
    cudaSetDevice(c->device);
    float* f[KIDMP_NFIELDS];
    if (layout == KIDMP_COL_FASTEST) {                // a column range of [nz][ncol] arrays: pitched copies
      for (int q = 0; q < KIDMP_NFIELDS; ++q) f[q] = fields[q] + c0;
      return step_pipelined(c, c1 - c0, nz, dt, f, p + c0, dz, ppt ? ppt + c0 : nullptr, ncol);
    }
    for (int q = 0; q < KIDMP_NFIELDS; ++q) f[q] = fields[q] + (size_t)c0 * nz;   // KiD's (k,i) arrays: a range of columns is contiguous
    std::vector<float> pp(ppt ? (size_t)(c1 - c0) * 4 : 0);
    if (kidmp_step(c, c1 - c0, nz, dt, layout, f, p + (size_t)c0 * nz, dz, ppt ? pp.data() : nullptr)) return 1;
    if (ppt) for (int q = 0; q < 4; ++q) memcpy(ppt + (size_t)q * ncol + c0, pp.data() + (size_t)q * (c1 - c0), (size_t)(c1 - c0) * 4);
    return 0;
  });
}

int multi_kid_interface(kidmp_handle* h, const kidmp_kid_columns* k, float dt, float p0, float r_on_cp) {
  MultiCtx* m = h->multi;
  const int n = (int)m->dev.size();
  if (!k->ppt) return fail(h, "kid_interface: null array");
  return on_all(h, [&](int d) -> int {
    long c0, c1;
    shard(k->nx, d, n, c0, c1);
    if (c1 <= c0) return 0;
    const size_t o = (size_t)c0 * k->nz;
    kidmp_kid_columns s = *k;                          // every array is (k,i): a range of columns is contiguous
    s.nx = c1 - c0;
    auto off = [&](const float* a) { return a ? a + o : nullptr; };
    auto offw = [&](float* a) { return a ? a + o : nullptr; };
    s.theta = off(k->theta); s.dtheta_adv = off(k->dtheta_adv); s.dtheta_div = off(k->dtheta_div); s.exner = off(k->exner);
    s.qv = off(k->qv); s.dqv_adv = off(k->dqv_adv); s.dqv_div = off(k->dqv_div);
    for (int q = 0; q < 7; ++q) {
      s.hyd[q] = off(k->hyd[q]); s.dhyd_adv[q] = off(k->dhyd_adv[q]); s.dhyd_div[q] = off(k->dhyd_div[q]);
      s.dhyd_mphys[q] = offw(k->dhyd_mphys[q]);
    }
    s.dtheta_mphys = offw(k->dtheta_mphys); s.dqv_mphys = offw(k->dqv_mphys);
    std::vector<float> pp((size_t)(c1 - c0) * 4);
    s.ppt = pp.data();
    if (kidmp_kid_interface(m->dev[d], &s, dt, p0, r_on_cp)) return 1;
    for (int q = 0; q < 4; ++q) memcpy(k->ppt + (size_t)q * k->nx + c0, pp.data() + (size_t)q * (c1 - c0), (size_t)(c1 - c0) * 4);
    return 0;
  });
}

int multi_diag(kidmp_handle* h, double out[KIDMP_NDIAG]) {
  DevRestore restore_;
  MultiCtx* m = h->multi;
  const int n = (int)m->dev.size();
  for (int d = 0; d < n; ++d) {                        // this device's sums, then cleared, as kidmp_diag does
    kidmp_handle* c = m->dev[d];
    cudaSetDevice(c->device);
    CK(h, cudaStreamWaitEvent(c->stream, c->ev_done, 0));
    CK(h, cudaMemcpyAsync(m->d_red[d], c->d_diag, KIDMP_NDIAG * 8, cudaMemcpyDeviceToDevice, c->stream));
    CK(h, cudaMemsetAsync(c->d_diag, 0, KIDMP_NDIAG * 8, c->stream));
  }
  int rc = m->GroupStart();
  for (int d = 0; d < n && !rc; ++d)                   // 64 bytes per device over NVLink: sum of the 8 f64 (ncclDouble = 8, ncclSum = 0)
    rc = m->AllReduce(m->d_red[d], m->d_red[d], KIDMP_NDIAG, 8, 0, m->comms[d], m->dev[d]->stream);
  const int rc2 = m->GroupEnd();
  if (rc || rc2) return fail(h, "diag: ncclAllReduce: %s", m->GetErrorString(rc ? rc : rc2));
  for (int d = 0; d < n; ++d) { cudaSetDevice(m->dev[d]->device); CK(h, cudaStreamSynchronize(m->dev[d]->stream)); }
  cudaSetDevice(m->dev[0]->device);
  CK(h, cudaMemcpy(out, m->d_red[0], KIDMP_NDIAG * 8, cudaMemcpyDeviceToHost));
  return 0;
}

int multi_init(const kidmp_config* cfg, kidmp_handle** out) {
  DevRestore restore_;
  kidmp_handle* h = new kidmp_handle();
  h->cfg = *cfg;
  MultiCtx* m = new MultiCtx();
  h->multi = m;
  auto bail = [&](const char* what) { g_init_error = std::string("kidmp_init: ") + what; kidmp_finalize(h); return 1; };
  std::vector<int> ids(cfg->ndev);
  for (int d = 0; d < cfg->ndev; ++d) {
    ids[d] = cfg->device_ids ? cfg->device_ids[d] : d;
    for (int e = 0; e < d; ++e) if (ids[e] == ids[d]) return bail("device_ids holds a device twice");
  }
  for (int d = 0; d < cfg->ndev; ++d) {
    kidmp_config one = *cfg;
    one.device = ids[d]; one.ndev = 0; one.device_ids = nullptr;
    kidmp_handle* c = nullptr;
    if (kidmp_init(&one, &c)) { const std::string w = g_init_error; return bail(w.c_str()); }
    m->dev.push_back(c);
  }
  h->device = ids[0];
  const char* path = getenv("KIDMP_NCCL_LIB");
  m->lib = dlopen(path ? path : "libnccl.so.2", RTLD_NOW | RTLD_LOCAL);
  if (!m->lib) return bail("ndev > 1 needs NCCL for the domain diagnostics: libnccl.so.2 not found (set KIDMP_NCCL_LIB)");
  m->CommInitAll = (int (*)(void**, int, const int*))dlsym(m->lib, "ncclCommInitAll");
  m->CommDestroy = (int (*)(void*))dlsym(m->lib, "ncclCommDestroy");
  m->AllReduce = (int (*)(const void*, void*, size_t, int, int, void*, cudaStream_t))dlsym(m->lib, "ncclAllReduce");
  m->GroupStart = (int (*)())dlsym(m->lib, "ncclGroupStart");
  m->GroupEnd = (int (*)())dlsym(m->lib, "ncclGroupEnd");
  m->GetErrorString = (const char* (*)(int))dlsym(m->lib, "ncclGetErrorString");
  if (!m->CommInitAll || !m->CommDestroy || !m->AllReduce || !m->GroupStart || !m->GroupEnd || !m->GetErrorString)
    return bail("the NCCL library lacks an entry point");
  m->comms.assign(cfg->ndev, nullptr);
  const int rc = m->CommInitAll(m->comms.data(), cfg->ndev, ids.data());
  if (rc) { m->comms.clear(); return bail(m->GetErrorString(rc)); }
  m->d_red.assign(cfg->ndev, nullptr);
  for (int d = 0; d < cfg->ndev; ++d) {
    cudaSetDevice(ids[d]);
    if (cudaMalloc((void**)&m->d_red[d], KIDMP_NDIAG * 8) != cudaSuccess) return bail("allocation failed");
  }
  *out = h;
  return 0;
}

void multi_finalize(kidmp_handle* h) {
  DevRestore restore_;
  MultiCtx* m = h->multi;
  for (size_t d = 0; d < m->d_red.size(); ++d) if (m->d_red[d]) { cudaSetDevice(m->dev[d]->device); cudaFree(m->d_red[d]); }
  for (void* c : m->comms) if (c && m->CommDestroy) m->CommDestroy(c);
  for (kidmp_handle* c : m->dev) kidmp_finalize(c);
  if (m->lib) dlclose(m->lib);
  delete m;
  delete h;
}

// resident state of a multi-device handle: every device holds its column range
int multi_state_alloc(kidmp_handle* h, long ncol, int nz) {
  MultiCtx* m = h->multi;
  const int n = (int)m->dev.size();
  if (ncol < n) return fail(h, "state_alloc: %ld columns over %d devices", ncol, n);
  for (int d = 0; d < n; ++d) {
    long c0, c1;
    shard(ncol, d, n, c0, c1);
    if (kidmp_state_alloc(m->dev[d], c1 - c0, nz)) return fail(h, "device %d: %s", m->dev[d]->device, m->dev[d]->err.c_str());
  }
  m->ncol = ncol; m->nz = nz;
  return 0;
}
int multi_copy(kidmp_handle* h, int layout, float* const fields[KIDMP_NFIELDS], const float* p, const float* dz, float* ppt, bool up) {
  MultiCtx* m = h->multi;
  const int n = (int)m->dev.size();
  if (!m->ncol) return fail(h, "upload / download before state_alloc");
  const long ncol = m->ncol;
  const int nz = m->nz;
  return on_all(h, [&](int d) -> int {
    kidmp_handle* c = m->dev[d];
    long c0, c1;
    shard(ncol, d, n, c0, c1);
    cudaSetDevice(c->device);
    const long w = c1 - c0;
    if (layout != KIDMP_COL_FASTEST) {                 // (k,i) arrays: a column range is contiguous
      float* f[KIDMP_NFIELDS];
      for (int q = 0; q < KIDMP_NFIELDS; ++q) f[q] = fields && fields[q] ? fields[q] + (size_t)c0 * nz : nullptr;
      if (up) return kidmp_upload(c, layout, f, p + (size_t)c0 * nz, dz);
      std::vector<float> pp(ppt ? (size_t)w * 4 : 0);
      if (kidmp_download(c, layout, fields ? f : nullptr, ppt ? pp.data() : nullptr)) return 1;
      if (ppt) for (int q = 0; q < 4; ++q) memcpy(ppt + (size_t)q * ncol + c0, pp.data() + (size_t)q * w, (size_t)w * 4);
      return 0;
    }
    const size_t hp = (size_t)ncol * 4, dp = (size_t)w * 4;
    for (int q = 0; q <= KIDMP_NFIELDS; ++q) {
      float* dev = field_ptr(c, q);
      if (up) {
        const float* src = (q < KIDMP_NFIELDS ? fields[q] : p) + c0;
        if (cudaMemcpy2DAsync(dev, dp, src, hp, dp, nz, cudaMemcpyHostToDevice, c->stream) != cudaSuccess) return fail(c, "upload failed");
      } else if (q < KIDMP_NFIELDS && fields && fields[q]) {
        if (cudaMemcpy2DAsync(fields[q] + c0, hp, dev, dp, dp, nz, cudaMemcpyDeviceToHost, c->stream) != cudaSuccess) return fail(c, "download failed");
      }
    }
    if (up && cudaMemcpyAsync(c->d_dz, dz, (size_t)nz * 4, cudaMemcpyHostToDevice, c->stream) != cudaSuccess) return fail(c, "upload failed");
    if (!up && ppt && cudaMemcpy2DAsync(ppt + c0, hp, c->d_ppt, dp, dp, 4, cudaMemcpyDeviceToHost, c->stream) != cudaSuccess) return fail(c, "download failed");
    return cudaStreamSynchronize(c->stream) == cudaSuccess ? 0 : fail(c, "copy failed");
  });
}
}  // namespace

extern "C" {

int kidmp_init(const kidmp_config* cfg, kidmp_handle** out) {
  if (!cfg || !out) return fail(nullptr, "kidmp_init: null argument");
  *out = nullptr;
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev < 1)
    return fail(nullptr, "kidmp_init: no CUDA device (%s); this library has no CPU path",
                e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
  if (!(cfg->set_Nc > 0.f)) return fail(nullptr, "kidmp_init: set_Nc must be positive");
  if (cfg->ndev > 1) {
    if (cfg->ndev > ndev) return fail(nullptr, "kidmp_init: ndev %d of %d devices", cfg->ndev, ndev);
    return multi_init(cfg, out);
  }
  const int dev1 = (cfg->ndev == 1 && cfg->device_ids) ? cfg->device_ids[0] : cfg->device;
  if (dev1 < 0 || dev1 >= ndev) return fail(nullptr, "kidmp_init: device %d of %d", dev1, ndev);
  kidmp_handle* h = new kidmp_handle();
  h->cfg = *cfg;
  h->device = dev1;
  if (getenv("KIDMP_CHUNK") && atol(getenv("KIDMP_CHUNK")) >= 32) h->chunk_cols = atol(getenv("KIDMP_CHUNK"));
  if (dev1 >= MAX_DEVICES) { delete h; return fail(nullptr, "kidmp_init: device ordinal %d not supported", dev1); }
  if (getenv("KIDMP_SIMPLE")) h->simple = atoi(getenv("KIDMP_SIMPLE")) != 0;
  if (getenv("KIDMP_GRAPHS")) h->graphs = atoi(getenv("KIDMP_GRAPHS")) != 0;
  if (getenv("KIDMP_GRAPH_MAX") && atol(getenv("KIDMP_GRAPH_MAX")) > 0) h->graph_max_cols = atol(getenv("KIDMP_GRAPH_MAX"));
  if (getenv("KIDMP_PIPE_CHUNK")) h->pipe_chunk = atol(getenv("KIDMP_PIPE_CHUNK")) > 1024 ? atol(getenv("KIDMP_PIPE_CHUNK")) : 1024;
  if (cfg->table_cache_path) h->cache_path = cfg->table_cache_path;
  h->cfg.table_cache_path = nullptr;
  auto bail = [&](int) { g_init_error = h->err; kidmp_finalize(h); return 1; };
  DevRestore restore_;
  if (cudaSetDevice(h->device) != cudaSuccess) { h->err = "cudaSetDevice failed"; return bail(1); }
  cudaDeviceProp prop;
  cudaGetDeviceProperties(&prop, h->device);
  h->nsm = prop.multiProcessorCount;
  if (prop.major < 10) { fail(h, "kidmp_init: built for sm_100a, device is sm_%d%d", prop.major, prop.minor); return bail(1); }
  // The second stream of a launch is made here, before the host makes its own: measured on the bench (a PyTorch stream made
  // after kidmp_init), a second stream made at the first step instead left k_substeps running 0.2 ms past k_finish.
  WorkSet& w = h->ws;
  if (cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreate(&h->ev0) != cudaSuccess || cudaEventCreate(&h->ev1) != cudaSuccess ||
      cudaEventCreateWithFlags(&h->ev_done, cudaEventDisableTiming) != cudaSuccess ||
      cudaStreamCreateWithFlags(&w.aux, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreateWithFlags(&w.ev_fork, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&w.ev_join, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&w.ev_lists_done, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&w.ev_n0_done, cudaEventDisableTiming) != cudaSuccess) {
    h->err = "stream/event creation failed"; return bail(1);
  }
  for (int q = 0; q <= KT_N; ++q) if (cudaEventCreate(&h->ev_k[q]) != cudaSuccess) {
    h->err = "stream/event creation failed"; return bail(1);
  }
  memset(&h->kc, 0, sizeof h->kc);
  memset(&h->hb, 0, sizeof h->hb);
  hostinit::Prep pp;
  hostinit::compute(h->cfg, h->kc, h->hb, pp);
  h->kc.t_Nc1 = h->hb.t_Nc[0];
  publish_constants(h);
  {
    // one slab for all lookup tables: one allocation, freed in one call
    size_t total = 0;
    for (auto& a : table_allocs(h)) total += (a.bytes + 255) / 256 * 256;
    if (cudaMalloc((void**)&h->d_tables, total) != cudaSuccess || cudaMemset(h->d_tables, 0, total) != cudaSuccess) {
      h->err = "table allocation failed"; return bail(1);
    }
    h->tables_bytes = total;
    size_t off = 0;
    for (auto& a : table_allocs(h)) { *a.p = h->d_tables + off; off += (a.bytes + 255) / 256 * 256; }
  }
  if (cudaMalloc((void**)&h->d_diag, KIDMP_NDIAG * 8) != cudaSuccess || cudaMemset(h->d_diag, 0, KIDMP_NDIAG * 8) != cudaSuccess) {
    h->err = "diag allocation failed"; return bail(1);
  }
  {
    static double et[KFM_N];
    static LogNode lt[KFM_N];
    kfm_build_tables(et, lt);
    if (cudaMemcpyToSymbol(g_exp_tab, et, sizeof et) != cudaSuccess || cudaMemcpyToSymbol(g_log_tab, lt, sizeof lt) != cudaSuccess) {
      h->err = "math table upload failed"; return bail(1);
    }
  }
  bool loaded = false;
  if (cfg->reuse_tables && !h->cache_path.empty()) loaded = load_cache(h) == 0;   // l_reuse_thompson_lookup, M:3720
  h->tables_from_cache = loaded;
  if (!loaded) {
    if (build_device_tables(h, pp)) return bail(1);
    if (cfg->reuse_tables && !h->cache_path.empty()) kidmp_save_tables(h, h->cache_path.c_str());
  }
  h->kc.racg = h->tabs.racg; h->kc.racs = h->tabs.racs; h->kc.qrfz = h->tabs.qrfz; h->kc.qcfz = h->tabs.qcfz;
  h->kc.iaus = h->tabs.iaus; h->kc.efrw = h->tabs.efrw; h->kc.efsw = h->tabs.efsw;
  *out = h;
  return 0;
}

int kidmp_finalize(kidmp_handle* h) {
  if (!h) return 0;
  if (h->multi) { multi_finalize(h); return 0; }
  DevGuard guard_(h->device);
  {
    std::lock_guard<std::mutex> lk(g_mu);
    if (g_const_owner[h->device] == h) g_const_owner[h->device] = nullptr;
  }
  // what this handle enqueued: steps end at ev_done (on whatever stream they ran), copies and staging on its own streams
  if (h->ev_done) cudaEventSynchronize(h->ev_done);
  for (cudaStream_t s : {h->stream, h->copy_in, h->copy_out}) if (s) cudaStreamSynchronize(s);
  free_state(h);
  for (auto& g : h->graph_cache) if (g.exec) cudaGraphExecDestroy(g.exec);
  if (h->d_tables) cudaFree(h->d_tables);
  if (h->d_tnc_wev) cudaFree(h->d_tnc_wev);
  if (h->d_aero) cudaFree(h->d_aero);
  if (h->d_partial) cudaFree(h->d_partial);
  if (h->d_diag) cudaFree(h->d_diag);
  if (h->d_kid) cudaFree(h->d_kid);
  if (h->h_kid) cudaFreeHost(h->h_kid);
  free_work(h->ws);
  for (cudaEvent_t e : {h->ws.ev_fork, h->ws.ev_join, h->ws.ev_lists_done, h->ws.ev_n0_done}) if (e) cudaEventDestroy(e);
  if (h->ws.aux) cudaStreamDestroy(h->ws.aux);
  for (int q = 0; q <= KT_N; ++q) if (h->ev_k[q]) cudaEventDestroy(h->ev_k[q]);
  if (h->ev_done) cudaEventDestroy(h->ev_done);
  if (h->d_pipe) cudaFree(h->d_pipe);
  if (h->d_pipe_dz) cudaFree(h->d_pipe_dz);
  if (h->h_ppt) cudaFreeHost(h->h_ppt);
  for (int b = 0; b < 3; ++b) for (int e = 0; e < 3; ++e) if (h->pipe_ev[b][e]) cudaEventDestroy(h->pipe_ev[b][e]);
  if (h->ev0) cudaEventDestroy(h->ev0);
  if (h->ev1) cudaEventDestroy(h->ev1);
  if (h->stream) cudaStreamDestroy(h->stream);
  if (h->copy_in) cudaStreamDestroy(h->copy_in);
  if (h->copy_out) cudaStreamDestroy(h->copy_out);
  delete h;
  return 0;
}

#ifndef KIDMP_BUILD_ID
#define KIDMP_BUILD_ID "00000000000000000000000000000000"
#endif
// hash of the sources and flags this binary was built from (kid_b200/build.py::source_id): ties the library to the tree
const char* kidmp_build_id(void) { static const char id[] = "KIDMP_BUILD_ID=" KIDMP_BUILD_ID; return id + 15; }

const char* kidmp_last_error(const kidmp_handle* h) { return h ? h->err.c_str() : g_init_error.c_str(); }
double kidmp_table_build_ms(const kidmp_handle* h) { if (h && h->multi) return kidmp_table_build_ms(h->multi->dev[0]); return h ? (double)h->table_ms : -1.0; }
int kidmp_tables_from_cache(const kidmp_handle* h) { if (h && h->multi) return kidmp_tables_from_cache(h->multi->dev[0]); return h && h->tables_from_cache ? 1 : 0; }

long kidmp_table_size(const kidmp_handle* h, const char* name) {
  if (!h || !name) return -1;
  if (h->multi) return kidmp_table_size(h->multi->dev[0], name);
  TabDesc d;
  if (find_table(h, name, d)) return d.n;
  auto it = h->consts.find(name);
  return it == h->consts.end() ? -1 : (long)it->second.size();
}

int kidmp_get_table(const kidmp_handle* hc, const char* name, double* out, long n) {
  kidmp_handle* h = const_cast<kidmp_handle*>(hc);
  if (!h || !name || !out) return 1;
  if (h->multi) return kidmp_get_table(h->multi->dev[0], name, out, n);
  TabDesc d;
  if (!find_table(h, name, d)) {
    auto it = h->consts.find(name);
    if (it == h->consts.end()) return fail(h, "unknown table '%s'", name);
    for (long i = 0; i < n && i < (long)it->second.size(); ++i) out[i] = it->second[i];
    return 0;
  }
  DevGuard guard_(h->device);
  CK(h, cudaStreamSynchronize(h->stream));
  const long m = n < d.n ? n : d.n;
  if (d.f32) {
    std::vector<float> tmp(d.n);
    CK(h, cudaMemcpy(tmp.data(), d.base, (size_t)d.n * 4, cudaMemcpyDeviceToHost));
    for (long i = 0; i < m; ++i) out[i] = (double)tmp[i];
  } else {
    std::vector<double> tmp((size_t)d.n * d.stride);
    CK(h, cudaMemcpy(tmp.data(), d.base, tmp.size() * 8, cudaMemcpyDeviceToHost));
    for (long i = 0; i < m; ++i) out[i] = tmp[(size_t)i * d.stride + d.member];
  }
  return 0;
}

int kidmp_save_tables(const kidmp_handle* hc, const char* path) {
  kidmp_handle* h = const_cast<kidmp_handle*>(hc);
  if (!h || !path) return 1;
  if (h->multi) return kidmp_save_tables(h->multi->dev[0], path);
  DevGuard guard_(h->device);
  CK(h, cudaStreamSynchronize(h->stream));
  const std::string tmp = std::string(path) + ".tmp";
  FILE* f = fopen(tmp.c_str(), "wb");
  if (!f) return fail(h, "cannot write %s", tmp.c_str());
  const uint64_t key = table_key(h);
  bool ok = fwrite(&key, 8, 1, f) == 1;
  std::vector<char> buf;
  for (auto& a : table_allocs(h)) {
    if (!ok) break;
    buf.resize(a.bytes);
    ok = cudaMemcpy(buf.data(), *a.p, a.bytes, cudaMemcpyDeviceToHost) == cudaSuccess &&
         fwrite(buf.data(), 1, a.bytes, f) == a.bytes;
  }
  fclose(f);
  if (!ok) { remove(tmp.c_str()); return fail(h, "writing %s failed", path); }
  if (rename(tmp.c_str(), path) != 0) return fail(h, "rename to %s failed", path);
  return 0;
}

// ---- KiD's list-directed text cache ------------------------------------------------------------------------------
namespace {
// one Fortran list-directed record per table, three values per line like gfortran's REAL(8) output
bool write_records(FILE* f, const std::vector<double>& rec, long n, int members) {
  for (int q = 0; q < members; ++q) {
    for (long i = 0; i < n; ++i) {
      if (fprintf(f, "%26.16E%s", rec[(size_t)i * members + q], (i % 3 == 2 || i == n - 1) ? "\n" : "") < 0) return false;
    }
  }
  return true;
}
// list-directed input: values separated by blanks, commas or line breaks; r*c repeats; D exponents
bool read_records(FILE* f, std::vector<double>& rec, long n, int members) {
  std::vector<char> tok;
  long have = 0;
  const long want = n * members;
  auto put = [&](double v, long rep) {
    for (long r = 0; r < rep && have < want; ++r, ++have) {
      const long q = have / n, i = have % n;          // records are table after table, elements in Fortran order
      rec[(size_t)i * members + q] = v;
    }
  };
  int c;
  while (have < want && (c = fgetc(f)) != EOF) {
    if (c == ' ' || c == ',' || c == '\n' || c == '\r' || c == '\t') continue;
    tok.clear();
    while (c != EOF && c != ' ' && c != ',' && c != '\n' && c != '\r' && c != '\t') { tok.push_back((char)((c == 'D' || c == 'd') ? 'E' : c)); c = fgetc(f); }
    tok.push_back(0);
    long rep = 1;
    char* star = strchr(tok.data(), '*');
    const char* val = tok.data();
    if (star) { *star = 0; rep = atol(tok.data()); val = star + 1; if (rep < 1) return false; }
    char* end = nullptr;
    const double v = strtod(val, &end);
    if (end == val) return false;
    put(v, rep);
  }
  return have == want;
}
}  // namespace

int kidmp_write_kid_cache(const kidmp_handle* hc, const char* racg_path, const char* racs_path) {
  kidmp_handle* h = const_cast<kidmp_handle*>(hc);
  if (!h || !racg_path || !racs_path) return 1;
  if (h->multi) return kidmp_write_kid_cache(h->multi->dev[0], racg_path, racs_path);
  if (h->kc.iiwarm) return fail(h, "write_kid_cache: the collection tables are not built when iiwarm (M:773)");
  DevGuard guard_(h->device);
  CK(h, cudaStreamSynchronize(h->stream));
  const struct { const char* path; const double* dev; long n; int members; } files[2] = {
      {racg_path, h->tabs.racg, (long)N_RACG, G_N}, {racs_path, h->tabs.racs, (long)N_RACS, S_N}};
  for (const auto& t : files) {
    std::vector<double> rec((size_t)t.n * t.members);
    CK(h, cudaMemcpy(rec.data(), t.dev, rec.size() * 8, cudaMemcpyDeviceToHost));
    // member order inside a record = order of the write statements (M:3823-3828, M:4066-4077)
    FILE* f = fopen(t.path, "w");
    if (!f) return fail(h, "cannot write %s", t.path);
    const bool ok = write_records(f, rec, t.n, t.members);
    if (fclose(f) != 0 || !ok) return fail(h, "writing %s failed", t.path);
  }
  return 0;
}

int kidmp_read_kid_cache(kidmp_handle* h, const char* racg_path, const char* racs_path) {
  if (!h || !racg_path || !racs_path) return 1;
  if (h->multi) {
    for (kidmp_handle* c : h->multi->dev) if (kidmp_read_kid_cache(c, racg_path, racs_path)) return fail(h, "%s", c->err.c_str());
    return 0;
  }
  if (h->kc.iiwarm) return fail(h, "read_kid_cache: the collection tables are not used when iiwarm (M:773)");
  DevGuard guard_(h->device);
  CK(h, cudaStreamSynchronize(h->stream));
  const struct { const char* path; double* dev; long n; int members; } files[2] = {
      {racg_path, h->tabs.racg, (long)N_RACG, G_N}, {racs_path, h->tabs.racs, (long)N_RACS, S_N}};
  for (const auto& t : files) {
    FILE* f = fopen(t.path, "r");
    if (!f) return fail(h, "cannot read %s", t.path);
    std::vector<double> rec((size_t)t.n * t.members);
    const bool ok = read_records(f, rec, t.n, t.members);
    fclose(f);
    if (!ok) return fail(h, "%s does not hold %d tables of %ld values", t.path, t.members, t.n);
    CK(h, cudaMemcpy(t.dev, rec.data(), rec.size() * 8, cudaMemcpyHostToDevice));
  }
  return 0;
}

int kidmp_state_alloc(kidmp_handle* h, long ncol, int nz) {
  if (!h) return 1;
  if (h->multi) return multi_state_alloc(h, ncol, nz);
  if (ncol < 1 || nz < 2 || nz > 256) return fail(h, "state_alloc: ncol=%ld nz=%d", ncol, nz);
  DevGuard guard_(h->device);
  if (h->ncol == ncol && h->nz == nz && h->d_state) return 0;
  free_state(h);
  const size_t n = (size_t)ncol * nz;
  CK(h, cudaMalloc((void**)&h->d_state, n * 4 * (KIDMP_NFIELDS + 1)));
  CK(h, cudaMalloc((void**)&h->d_stage, n * 4));
  CK(h, cudaMalloc((void**)&h->d_dz, (size_t)nz * 4));
  CK(h, cudaMalloc((void**)&h->d_ppt, (size_t)ncol * 4 * 4));
  CK(h, cudaMemset(h->d_ppt, 0, (size_t)ncol * 4 * 4));
  if (h->rates_on) CK(h, cudaMalloc((void**)&h->d_rates_own, n * KIDMP_NRATES * 4));
  h->ncol = ncol; h->nz = nz;
  return 0;
}

int kidmp_enable_rates(kidmp_handle* h, int on) {
  if (!h) return 1;
  if (h->multi) {
    for (kidmp_handle* c : h->multi->dev) if (kidmp_enable_rates(c, on)) return fail(h, "%s", c->err.c_str());
    return 0;
  }
  DevGuard guard_(h->device);
  h->rates_on = on != 0;
  if (!h->rates_on && h->d_rates_own) { CK(h, cudaEventSynchronize(h->ev_done)); cudaFree(h->d_rates_own); h->d_rates_own = nullptr; }
  if (h->rates_on && !h->d_rates_own && h->d_state)
    CK(h, cudaMalloc((void**)&h->d_rates_own, (size_t)h->ncol * h->nz * KIDMP_NRATES * 4));
  return 0;
}

int kidmp_get_rates(kidmp_handle* h, int layout, float* rates) {
  if (!h || !rates) return 1;
  if (h->multi) {
    MultiCtx* m = h->multi;
    if (layout != KIDMP_K_FASTEST) return fail(h, "get_rates: a multi-device handle returns KIDMP_K_FASTEST rates");
    const int n = (int)m->dev.size();
    for (int d = 0; d < n; ++d) {
      kidmp_handle* c = m->dev[d];
      if (!c->d_rates_own) return fail(h, "get_rates: kidmp_enable_rates and a step first");
      long c0, c1;
      shard(m->ncol ? m->ncol : c->ncol, d, n, c0, c1);
      std::vector<float> part((size_t)KIDMP_NRATES * c->ncol * c->nz);
      if (kidmp_get_rates(c, layout, part.data())) return fail(h, "%s", c->err.c_str());
      const long total = m->ncol ? m->ncol : c->ncol;
      for (int r = 0; r < KIDMP_NRATES; ++r)
        memcpy(rates + ((size_t)r * total + c0) * c->nz, part.data() + (size_t)r * c->ncol * c->nz, (size_t)c->ncol * c->nz * 4);
    }
    return 0;
  }
  if (!h->d_rates_own || !h->d_state) return fail(h, "get_rates: kidmp_enable_rates and a step on the resident state first");
  DevGuard guard_(h->device);
  const size_t n = (size_t)h->ncol * h->nz;
  CK(h, cudaStreamWaitEvent(h->stream, h->ev_done, 0));
  if (layout == KIDMP_COL_FASTEST || h->ncol == 1) {
    CK(h, cudaMemcpyAsync(rates, h->d_rates_own, n * KIDMP_NRATES * 4, cudaMemcpyDeviceToHost, h->stream));
  } else {
    dim3 g((unsigned)((h->ncol + 31) / 32), (unsigned)((h->nz + 31) / 32)), b(32, 8);
    for (int r = 0; r < KIDMP_NRATES; ++r) {           // [nz][ncol] -> KiD's (k,i) order, plane by plane through the staging buffer
      k_transpose<<<g, b, 0, h->stream>>>(h->d_rates_own + n * r, h->d_stage, h->ncol, h->nz, 0);
      ++h->launches;
      CK(h, cudaMemcpyAsync(rates + n * r, h->d_stage, n * 4, cudaMemcpyDeviceToHost, h->stream));
      CK(h, cudaStreamSynchronize(h->stream));
    }
  }
  CK(h, cudaStreamSynchronize(h->stream));
  return 0;
}

int kidmp_upload(kidmp_handle* h, int layout, const float* const fields[KIDMP_NFIELDS], const float* p, const float* dz) {
  if (h && h->multi) {
    if (!fields || !p || !dz) return fail(h, "upload: null pointer");
    for (int q = 0; q < KIDMP_NFIELDS; ++q) if (!fields[q]) return fail(h, "upload: field %d is null", q);
    return multi_copy(h, layout, const_cast<float* const*>(fields), p, dz, nullptr, true);
  }
  if (!h || !h->d_state) return h ? fail(h, "upload before state_alloc") : 1;
  if (!fields || !p || !dz) return fail(h, "upload: null pointer");
  DevGuard guard_(h->device);
  for (int q = 0; q < KIDMP_NFIELDS; ++q) {
    if (!fields[q]) return fail(h, "upload: field %d is null", q);
    if (put_field(h, layout, fields[q], field_ptr(h, q))) return 1;
    if (layout != KIDMP_COL_FASTEST && h->ncol > 1) CK(h, cudaStreamSynchronize(h->stream));
  }
  if (put_field(h, layout, p, field_ptr(h, KIDMP_NFIELDS))) return 1;
  CK(h, cudaMemcpyAsync(h->d_dz, dz, (size_t)h->nz * 4, cudaMemcpyHostToDevice, h->stream));
  CK(h, cudaStreamSynchronize(h->stream));
  return 0;
}

int kidmp_step_resident(kidmp_handle* h, float dt) {
  if (h && h->multi) {
    for (kidmp_handle* c : h->multi->dev) if (kidmp_step_resident(c, dt)) return fail(h, "device %d: %s", c->device, c->err.c_str());
    return 0;                                           // asynchronous on every device, like the single-device call
  }
  if (!h || !h->d_state) return h ? fail(h, "step before state_alloc") : 1;
  DevGuard guard_(h->device);
  CK(h, cudaEventRecord(h->ev0, h->stream));
  if (launch_step(h, resident_args(h, dt), h->stream)) return 1;
  CK(h, cudaEventRecord(h->ev1, h->stream));
  return 0;
}

int kidmp_download(kidmp_handle* h, int layout, float* const fields[KIDMP_NFIELDS], float* ppt) {
  if (h && h->multi) return multi_copy(h, layout, fields, nullptr, nullptr, ppt, false);
  if (!h || !h->d_state) return h ? fail(h, "download before state_alloc") : 1;
  DevGuard guard_(h->device);
  if (fields)
    for (int q = 0; q < KIDMP_NFIELDS; ++q)
      if (fields[q] && get_field(h, layout, field_ptr(h, q), fields[q])) return 1;
  if (ppt) CK(h, cudaMemcpyAsync(ppt, h->d_ppt, (size_t)h->ncol * 16, cudaMemcpyDeviceToHost, h->stream));
  CK(h, cudaStreamSynchronize(h->stream));
  return 0;
}

// Large column-fastest domains: the columns are cut into chunks that flow through three streams
// (H2D copy, the two step kernels, D2H copy) on double buffers, so both PCIe directions and the
// SMs work at the same time.  Columns are independent, so chunking does not change any result.
// `hld`: columns of the caller's host arrays (their row stride): a multi-device handle gives every device a range of columns
// of the same arrays.
static int step_pipelined(kidmp_handle* h, long ncol, int nz, float dt, float* const fields[KIDMP_NFIELDS],
                          const float* p, const float* dz, float* ppt, long hld) {
  // (no larger than a launch chunk: then every pipeline chunk is one launch of launch_step, whose column flags k_scatter_host reads)
  const long chunk = h->pipe_chunk < h->chunk_cols ? h->pipe_chunk : h->chunk_cols;
  const int NB = 3;
  // (streams are made when they are first needed: the device has few hardware queues, and streams that share one
  // serialise kernels that could run side by side)
  if (!h->copy_in) CK(h, cudaStreamCreateWithFlags(&h->copy_in, cudaStreamNonBlocking));
  if (!h->copy_out) CK(h, cudaStreamCreateWithFlags(&h->copy_out, cudaStreamNonBlocking));
  const size_t cells = (size_t)chunk * nz;
  const size_t per_buf = cells * (KIDMP_NFIELDS + 1) + (size_t)chunk * 4;
  if (h->pipe_floats < per_buf * NB || h->pipe_nz != nz) {
    if (h->d_pipe) cudaFree(h->d_pipe);
    h->d_pipe = nullptr; h->pipe_floats = 0;
    CK(h, cudaMalloc((void**)&h->d_pipe, per_buf * NB * 4));
    h->pipe_floats = per_buf * NB; h->pipe_nz = nz;
    if (!h->d_pipe_dz) CK(h, cudaMalloc((void**)&h->d_pipe_dz, 256 * 4));
    for (int b = 0; b < NB; ++b)
      for (int e = 0; e < 3; ++e)
        if (!h->pipe_ev[b][e]) CK(h, cudaEventCreateWithFlags(&h->pipe_ev[b][e], cudaEventDisableTiming));
  }
  // ppt goes through a pinned staging buffer: a D2H copy into pageable memory would block the host at every
  // chunk and serialise the pipeline
  if (ppt && h->h_ppt_floats < (size_t)ncol * 4) {
    if (h->h_ppt) cudaFreeHost(h->h_ppt);
    h->h_ppt = nullptr; h->h_ppt_floats = 0;
    CK(h, cudaHostAlloc((void**)&h->h_ppt, (size_t)ncol * 16, cudaHostAllocDefault));
    h->h_ppt_floats = (size_t)ncol * 4;
  }
  CK(h, cudaMemcpyAsync(h->d_pipe_dz, dz, (size_t)nz * 4, cudaMemcpyHostToDevice, h->stream));
  CK(h, cudaEventRecord(h->ev0, h->stream));
  // Pinned output arrays (cudaHostAlloc / cudaHostRegister: what a host that cares about transfer speed uses): only the
  // columns the step changed go back, written by a kernel straight into the host arrays (k_scatter_host); pageable arrays
  // get the whole chunk back with a copy.  KIDMP_ZEROCOPY=0 switches the first path off.
  HostFields hf{};
  bool zero_copy = !(getenv("KIDMP_ZEROCOPY") && atoi(getenv("KIDMP_ZEROCOPY")) == 0);
  for (int q = 0; q < KIDMP_NFIELDS && zero_copy; ++q) {
    cudaPointerAttributes at{};
    if (cudaPointerGetAttributes(&at, fields[q]) != cudaSuccess || at.type != cudaMemoryTypeHost || !at.devicePointer) { zero_copy = false; cudaGetLastError(); }
    else hf.f[q] = (float*)at.devicePointer;
  }
  h->last_zero_copy = zero_copy;
  const size_t hpitch = (size_t)hld * 4, ppitch = (size_t)ncol * 4;
  // KIDMP_PIPE_TRACE=1: device timeline of every chunk (H2D, step kernels, return path) on stderr after the step
  const bool trace = getenv("KIDMP_PIPE_TRACE") && atoi(getenv("KIDMP_PIPE_TRACE")) != 0;
  std::vector<cudaEvent_t> tev;
  auto tmark = [&](cudaStream_t st) { if (trace) { cudaEvent_t e; cudaEventCreate(&e); cudaEventRecord(e, st); tev.push_back(e); } };
  long c0 = 0;
  for (int it = 0; c0 < ncol; ++it, c0 += chunk) {
    const int b = it % NB;
    const long n = (ncol - c0 < chunk) ? (ncol - c0) : chunk;
    float* base = h->d_pipe + per_buf * b;
    float* d_ppt = base + cells * (KIDMP_NFIELDS + 1);
    const size_t dpitch = (size_t)n * 4;
    if (it >= NB) CK(h, cudaStreamWaitEvent(h->copy_in, h->pipe_ev[b][2], 0));     // buffer drained by its D2H
    tmark(h->copy_in);
    for (int q = 0; q <= KIDMP_NFIELDS; ++q) {
      const float* src = (q < KIDMP_NFIELDS ? fields[q] : p) + c0;
      CK(h, cudaMemcpy2DAsync(base + cells * q, dpitch, src, hpitch, dpitch, nz, cudaMemcpyHostToDevice, h->copy_in));
    }
    CK(h, cudaEventRecord(h->pipe_ev[b][0], h->copy_in));
    tmark(h->copy_in);
    CK(h, cudaStreamWaitEvent(h->stream, h->pipe_ev[b][0], 0));
    tmark(h->stream);
    StepArgs a{};
    a.ncol = n; a.ld = n; a.nz = nz; a.dt = dt;
    for (int q = 0; q < KIDMP_NFIELDS; ++q) a.f[q] = base + cells * q;
    a.p = base + cells * KIDMP_NFIELDS; a.dz = h->d_pipe_dz; a.ppt = d_ppt;
    if (launch_step(h, a, h->stream)) return 1;
    tmark(h->stream);
    CK(h, cudaEventRecord(h->pipe_ev[b][1], h->stream));
    CK(h, cudaStreamWaitEvent(h->copy_out, h->pipe_ev[b][1], 0));
    if (zero_copy) {
      HostFields hc = hf;
      for (int q = 0; q < KIDMP_NFIELDS; ++q) hc.f[q] += c0;
      StepArgs sa = a;
      sa.colflag = h->ws.d_colflag;                  // (this chunk's flags: it was one launch, and the next chunk's kernels follow on this stream)
      k_scatter_host<<<(unsigned)((n + 127) / 128), 128, 0, h->stream>>>(sa, hc, hld);
      ++h->launches;
      CK(h, cudaEventRecord(h->pipe_ev[b][1], h->stream));
      CK(h, cudaStreamWaitEvent(h->copy_out, h->pipe_ev[b][1], 0));
    } else
      for (int q = 0; q < KIDMP_NFIELDS; ++q)
        CK(h, cudaMemcpy2DAsync(fields[q] + c0, hpitch, base + cells * q, dpitch, dpitch, nz, cudaMemcpyDeviceToHost, h->copy_out));
    if (ppt) CK(h, cudaMemcpy2DAsync(h->h_ppt + c0, ppitch, d_ppt, dpitch, dpitch, 4, cudaMemcpyDeviceToHost, h->copy_out));
    CK(h, cudaEventRecord(h->pipe_ev[b][2], h->copy_out));
    tmark(h->stream);
    tmark(h->copy_out);
  }
  CK(h, cudaEventRecord(h->ev1, h->stream));
  CK(h, cudaStreamSynchronize(h->copy_out));
  CK(h, cudaStreamSynchronize(h->stream));
  if (trace) {
    fprintf(stderr, "chunk  h2d_start h2d_end  step_start step_end  return_end(stream) return_end(copy_out)   [ms from the first H2D]\n");
    for (size_t i = 0; i + 5 < tev.size() + 1 && i + 5 < tev.size() + 6 && i + 6 <= tev.size(); i += 6) {
      float t[6];
      for (int j = 0; j < 6; ++j) cudaEventElapsedTime(&t[j], tev[0], tev[i + j]);
      fprintf(stderr, "%5zu  %8.2f %8.2f  %8.2f %8.2f  %8.2f %8.2f\n", i / 6, t[0], t[1], t[2], t[3], t[4], t[5]);
    }
    for (cudaEvent_t e : tev) cudaEventDestroy(e);
  }
  if (ppt) for (int q = 0; q < 4; ++q) memcpy(ppt + (size_t)q * hld, h->h_ppt + (size_t)q * ncol, (size_t)ncol * 4);
  return 0;
}

int kidmp_step(kidmp_handle* h, long ncol, int nz, float dt, int layout, float* const fields[KIDMP_NFIELDS],
               const float* p, const float* dz, float* ppt) {
  if (!h) return 1;
  if (ncol == 0) return 0;                               // `do i = 1, nx` with nx = 0 (I:54): nothing to do, nothing touched
  if (!fields || !p || !dz) return fail(h, "step: null pointer");
  if (h->multi) return multi_step(h, ncol, nz, dt, layout, fields, p, dz, ppt);
  // (with a process-rate buffer set the whole domain goes through the resident path: the buffer is [36][nz][ncol] of the domain)
  if (layout == KIDMP_COL_FASTEST && ncol >= 2 * h->pipe_chunk && nz >= 2 && nz <= 256 && dt > 0.f && !h->d_rates) {
    for (int q = 0; q < KIDMP_NFIELDS; ++q) if (!fields[q]) return fail(h, "step: field %d is null", q);
    DevGuard guard_(h->device);
    return step_pipelined(h, ncol, nz, dt, fields, p, dz, ppt, ncol);
  }
  if (kidmp_state_alloc(h, ncol, nz)) return 1;
  if (kidmp_upload(h, layout, fields, p, dz)) return 1;
  if (kidmp_step_resident(h, dt)) return 1;
  return kidmp_download(h, layout, fields, ppt);
}

int kidmp_column(kidmp_handle* h, int nz, float dt, float* qv, float* qc, float* qi, float* qr, float* qs, float* qg,
                 float* ni, float* nr, float* t, const float* p, const float* dz, float* ppt4) {
  if (!h) return 1;
  if (h->multi) return kidmp_column(h->multi->dev[0], nz, dt, qv, qc, qi, qr, qs, qg, ni, nr, t, p, dz, ppt4) ? fail(h, "%s", h->multi->dev[0]->err.c_str()) : 0;
  if (!ppt4) return fail(h, "column: ppt4 is null");
  float* f[KIDMP_NFIELDS] = {qv, qc, qi, qr, qs, qg, ni, nr, t};
  float inc[4] = {0.f, 0.f, 0.f, 0.f};
  if (kidmp_step(h, 1, nz, dt, KIDMP_K_FASTEST, f, p, dz, inc)) return 1;
  for (int q = 0; q < 4; ++q) ppt4[q] = ppt4[q] + inc[q];   // INOUT accumulators, M:1172
  return 0;
}

int kidmp_step_device(kidmp_handle* h, long ncol, int nz, float dt, float* const d_fields[KIDMP_NFIELDS],
                      const float* d_p, const float* d_dz, float* d_ppt, void* stream) {
  if (!h) return 1;
  if (h->multi) return fail(h, "step_device: device pointers belong to one device; use a single-device handle per GPU");
  if (ncol == 0) return 0;
  if (!d_fields || !d_p || !d_dz || !d_ppt) return fail(h, "step_device: null pointer");
  DevGuard guard_(h->device);
  StepArgs a{};
  a.ncol = ncol; a.ld = ncol; a.nz = nz; a.dt = dt; a.rates = h->d_rates;
  for (int q = 0; q < KIDMP_NFIELDS; ++q) { if (!d_fields[q]) return fail(h, "step_device: field %d is null", q); a.f[q] = d_fields[q]; }
  a.p = d_p; a.dz = d_dz; a.ppt = d_ppt;
  cudaStream_t s = stream ? (cudaStream_t)stream : h->stream;
  if (s == h->stream) CK(h, cudaEventRecord(h->ev0, s));
  if (launch_step(h, a, s)) return 1;
  if (s == h->stream) CK(h, cudaEventRecord(h->ev1, s));
  return 0;
}

// table_dropEvap, M:4400-4439: number of the cloud droplets smaller than D-star for every (D-star bin, cloud water node,
// droplet number node).  Only an aerosol-aware run reads it (M:2850): built by the first such step - slope and intercept of the
// 3 700 spectra on the host (two powers each, like the per-node scalars of the other tables), the 370 000 bin sums by
// k_table_wev - and the constants re-published.
int ensure_wev_table(kidmp_handle* h) {
  if (h->d_tnc_wev) return 0;
  const HostBins& b = h->hb;
  const KConst& kc = h->kc;
  std::vector<double> lamc((size_t)NTB_C * NBINS), N0_c((size_t)NTB_C * NBINS);
  std::vector<int> nu(NBINS);
  for (int k = 0; k < NBINS; ++k) {
    const int nu_c = std::min(15, (int)std::lround((double)1000.E6f / b.t_Nc[k]) + 2);
    nu[k] = nu_c;
    for (int j = 0; j < NTB_C; ++j) {
      const double l = std::pow(b.t_Nc[k] * (double)kc.am_r * (double)kc.ccg[1][nu_c - 1] * (double)kc.ocg1[nu_c - 1] / (double)b.r_c[j], (double)kc.obmr);
      lamc[j + (size_t)NTB_C * k] = l;
      N0_c[j + (size_t)NTB_C * k] = b.t_Nc[k] * (double)kc.ocg1[nu_c - 1] * std::pow(l, (double)kc.cce[0][nu_c - 1]);
    }
  }
  std::vector<void*> keep;
  const double *d_lamc = nullptr, *d_N0 = nullptr, *d_Dc = nullptr, *d_dtc = nullptr;
  const int* d_nu = nullptr;
  cudaError_t e = to_dev(lamc, &d_lamc, keep);
  if (e == cudaSuccess) e = to_dev(N0_c, &d_N0, keep);
  if (e == cudaSuccess) e = to_dev(nu, &d_nu, keep);
  if (e == cudaSuccess) e = to_dev(b.Dc, NBINS, &d_Dc, keep);
  if (e == cudaSuccess) e = to_dev(b.dtc, NBINS, &d_dtc, keep);
  if (e == cudaSuccess) e = cudaMalloc((void**)&h->d_tnc_wev, (size_t)NBINS * NTB_C * NBINS * 8);
  if (e == cudaSuccess) {
    k_table_wev<<<NTB_C * NBINS, 128, 0, h->stream>>>(d_lamc, d_N0, d_nu, d_Dc, d_dtc, h->d_tnc_wev);
    ++h->launches;
    e = cudaStreamSynchronize(h->stream);
    if (e == cudaSuccess) e = cudaGetLastError();
  }
  for (void* q : keep) cudaFree(q);
  if (e != cudaSuccess) { if (h->d_tnc_wev) { cudaFree(h->d_tnc_wev); h->d_tnc_wev = nullptr; } return fail(h, "table_dropEvap: %s", cudaGetErrorString(e)); }
  h->kc.tnc_wev = h->d_tnc_wev;
  std::lock_guard<std::mutex> lk(g_mu);
  if (g_const_owner[h->device] == h) g_const_owner[h->device] = nullptr;      // the next step uploads the constants again
  return 0;
}

int kidmp_step_device_aero(kidmp_handle* h, long ncol, int nz, float dt, float* const d_fields[KIDMP_NFIELDS], float* d_nc,
                           float* d_nwfa, float* d_nifa, const float* d_p, const float* d_w, const float* d_dz,
                           const float* d_nwfa2d, float* d_ppt, void* stream) {
  if (!h) return 1;
  if (h->multi) return fail(h, "step_device_aero: device pointers belong to one device; use a single-device handle per GPU");
  if (ncol == 0) return 0;
  if (!d_fields || !d_nc || !d_nwfa || !d_nifa || !d_p || !d_w || !d_dz || !d_ppt) return fail(h, "step_device_aero: null pointer");
  if (h->d_rates || h->rates_on) return fail(h, "step_device_aero: the process-rate buffer is not available in an aerosol-aware step");
  DevGuard guard_(h->device);
  if (ensure_wev_table(h)) return 1;
  StepArgs a{};
  a.ncol = ncol; a.ld = ncol; a.nz = nz; a.dt = dt;
  for (int q = 0; q < KIDMP_NFIELDS; ++q) { if (!d_fields[q]) return fail(h, "step_device_aero: field %d is null", q); a.f[q] = d_fields[q]; }
  a.p = d_p; a.dz = d_dz; a.ppt = d_ppt; a.nc = d_nc; a.nwfa = d_nwfa; a.nifa = d_nifa; a.w = d_w;
  cudaStream_t s = stream ? (cudaStream_t)stream : h->stream;
  if (s == h->stream) CK(h, cudaEventRecord(h->ev0, s));
  if (launch_step(h, a, s)) return 1;
  // what mp_gt_driver does after the call (M:1001): surface emission into the lowest level, every column
  if (d_nwfa2d) { k_nwfa_surface<<<(unsigned)((ncol + 255) / 256), 256, 0, s>>>(d_nwfa, d_nwfa2d, ncol, dt); ++h->launches; CK(h, cudaEventRecord(h->ev_done, s)); }
  if (s == h->stream) CK(h, cudaEventRecord(h->ev1, s));
  return 0;
}

int kidmp_set_rates_buffer(kidmp_handle* h, float* d_rates) {
  if (!h) return 1;
  if (h->multi) return fail(h, "set_rates_buffer: device pointers belong to one device; use a single-device handle");
  h->d_rates = d_rates;
  return 0;
}

const char* kidmp_rate_names(void) {
  return "pri_inu,pri_ide,prs_ide,prs_sde,prg_gde,pri_wfz,prs_scw,prg_scw,prg_gcw,pri_ihm,pri_rfz,prs_iau,"
         "prs_sci,pri_rci,pni_inu,pni_ihm,pni_wfz,pni_rfz,pni_ide,pni_iau,pni_sci,pni_rci,prr_sml,prr_gml,"
         "pnr_rcs,pnr_rcg,pnr_rci,pnr_sml,pnr_gml,pnr_rfz,prr_wau,prr_rcw,prv_rev,pnr_wau,pnr_rev,pnr_rcr";
}

int kidmp_diag(kidmp_handle* h, double out[KIDMP_NDIAG]) {
  if (!h || !out) return 1;
  if (h->multi) return multi_diag(h, out);
  DevGuard guard_(h->device);
  CK(h, cudaStreamWaitEvent(h->stream, h->ev_done, 0));   // the last step may have run on a caller's stream
  CK(h, cudaMemcpyAsync(out, h->d_diag, KIDMP_NDIAG * 8, cudaMemcpyDeviceToHost, h->stream));
  CK(h, cudaMemsetAsync(h->d_diag, 0, KIDMP_NDIAG * 8, h->stream));
  CK(h, cudaStreamSynchronize(h->stream));
  return 0;
}

// mp_gt_driver, M:806-1143 (see kidmp_wrf.cuh).  Every entry is one tile of the caller's memory box; the packed entries
// step the whole box.  One set of kernels serves both sides: the device entry runs them on the caller's arrays, the host
// entry stages the tile rows through the pinned buffer and runs them on the packed tile (a box of its own).
int kidmp_mp_gt_driver(kidmp_handle* h, const kidmp_wrf_fields* w, float dt_in) {
  if (!h) return 1;
  if (!w) return fail(h, "mp_gt_driver: null argument");
  const kidmp_wrf_tile t{0, w->ni, 0, w->nk, 0, w->nj};
  return kidmp_mp_gt_driver_tile(h, w, &t, nullptr, dt_in);
}
int kidmp_mp_gt_driver_aero(kidmp_handle* h, const kidmp_wrf_fields* w, const kidmp_wrf_aerosols* ae, float dt_in) {
  if (!h) return 1;
  if (!ae) return fail(h, "mp_gt_driver_aero: null aerosol array");
  if (!w) return fail(h, "mp_gt_driver: null argument");
  const kidmp_wrf_tile t{0, w->ni, 0, w->nk, 0, w->nj};
  return kidmp_mp_gt_driver_tile(h, w, &t, ae, dt_in);
}

// Every check of a tile call, before anything is copied or launched: a rejected call leaves every array as it was.
static int wrf_check(kidmp_handle* h, const char* who, const kidmp_wrf_fields* w, const kidmp_wrf_tile* t,
                     const kidmp_wrf_aerosols* ae, float dt_in) {
  if (!w || !t) return fail(h, "%s: null argument", who);
  if (w->ni < 1 || w->nj < 1 || w->nk < 2) return fail(h, "%s: bad memory dimensions %d x %d x %d", who, w->ni, w->nk, w->nj);
  if (t->ni < 1 || t->nj < 1 || t->nk < 2 || t->nk > 256)
    return fail(h, "%s: bad tile extents %d x %d x %d (ni, nj >= 1, 2 <= nk <= 256)", who, t->ni, t->nk, t->nj);
  if (t->i0 < 0 || t->k0 < 0 || t->j0 < 0 || (long)t->i0 + t->ni > w->ni || (long)t->k0 + t->nk > w->nk || (long)t->j0 + t->nj > w->nj)
    return fail(h, "%s: tile i %d+%d, k %d+%d, j %d+%d does not lie inside the memory box %d x %d x %d", who, t->i0, t->ni,
                t->k0, t->nk, t->j0, t->nj, w->ni, w->nk, w->nj);
  if (t->nj > 65535) return fail(h, "%s: tile nj = %d, at most 65535", who, t->nj);
  const float* const io[9] = {w->qv, w->qc, w->qi, w->qr, w->qs, w->qg, w->ni_, w->nr, w->th};
  for (int q = 0; q < 9; ++q) if (!io[q]) return fail(h, "%s: null field %d", who, q);
  if (!w->pii || !w->p || !w->dz || !w->rainnc || !w->rainncv || !w->sr) return fail(h, "%s: null array", who);
  if (!(dt_in > 0.f)) return fail(h, "%s: dt must be positive", who);
  if (ae) {
    if (!ae->nc || !ae->nwfa || !ae->nifa || !ae->w) return fail(h, "%s: null aerosol array", who);
    if (h->d_rates || h->rates_on) return fail(h, "%s: the process-rate buffer is not available in an aerosol-aware step", who);
  }
  return 0;
}

static int ensure_dev(kidmp_handle* h, float** p, size_t* have, size_t need) {
  if (*have >= need) return 0;
  if (*p) cudaFree(*p);
  *p = nullptr; *have = 0;
  CK(h, cudaMalloc((void**)p, need * 4));
  *have = need;
  return 0;
}

// The kernels of one call on device arrays that a.t addresses, on stream s: the tile into the resident planes, the step,
// the planes back into the tile, the accumulators.  ae4: nc nwfa nifa w of an aerosol-aware call (else NULL), nwfa2d or NULL,
// with their planes in h->d_aero.  The caller sets a.t, the tile's arrays and a.dz_col; a.f, a.p, a.ppt are set here.
static int wrf_kernels(kidmp_handle* h, WrfArgs& a, float* const* ae4, const float* nwfa2d, float dt_in, cudaStream_t s) {
  const long ncol = (long)a.t.ni * a.t.nj;
  const size_t n = (size_t)ncol * a.t.nk;
  if (ae4 && ensure_wev_table(h)) return 1;
  for (int q = 0; q < KIDMP_NFIELDS; ++q) a.f[q] = field_ptr(h, q);
  a.p = field_ptr(h, KIDMP_NFIELDS);
  a.ppt = h->d_ppt;
  CK(h, cudaStreamWaitEvent(s, h->ev_done, 0));         // the resident planes and staging may serve a step on another stream
  const dim3 b(128), g((unsigned)((a.t.ni + 127) / 128), (unsigned)a.t.nk, (unsigned)a.t.nj);
  const dim3 g2(g.x, 1, g.z);
  WrfBox t2 = a.t;                                      // the (i,j) arrays: a box of one level
  t2.nk = 1; t2.nk_m = 1; t2.k0 = 0;
  k_wrf_gather<<<g, b, 0, s>>>(a);
  if (s == h->stream) CK(h, cudaEventRecord(h->ev0, s));
  StepArgs sa = resident_args(h, dt_in);
  sa.dz_col = a.dz_col;
  float* const d_ae = h->d_aero;                         // aerosol-aware run: 4 planes and the nwfa2d plane
  if (ae4) {
    for (int q = 0; q < 4; ++q) k_ikj_planes<<<g, b, 0, s>>>(ae4[q], d_ae + n * q, a.t, 1);
    if (nwfa2d) k_ikj_planes<<<g2, b, 0, s>>>(const_cast<float*>(nwfa2d), d_ae + 4 * n, t2, 1);   // (read only)
    sa.nc = d_ae; sa.nwfa = d_ae + n; sa.nifa = d_ae + 2 * n; sa.w = d_ae + 3 * n;
    a.nc_plane = sa.nc;
    h->launches += nwfa2d ? 5 : 4;
  }
  if (launch_step(h, sa, s)) return 1;
  if (ae4 && nwfa2d) { k_nwfa_surface<<<(unsigned)((ncol + 255) / 256), 256, 0, s>>>(sa.nwfa, d_ae + 4 * n, ncol, dt_in); ++h->launches; }   // M:1001
  if (s == h->stream) CK(h, cudaEventRecord(h->ev1, s));
  k_wrf_scatter<<<g, b, 0, s>>>(a, h->kc.Nt_c);
  if (ae4) {
    for (int q = 0; q < 3; ++q) k_ikj_planes<<<g, b, 0, s>>>(ae4[q], d_ae + n * q, a.t, 0);
    h->launches += 3;
  }
  k_wrf_accumulate<<<(unsigned)((ncol + 255) / 256), 256, 0, s>>>(a);
  h->launches += 3;
  CK(h, cudaGetLastError());
  CK(h, cudaEventRecord(h->ev_done, s));                 // the next call or kidmp_diag reuses the planes, maybe on another stream
  return 0;
}

// the tile rows of one array between the caller's memory box `mem` (ni_m x nk_m x ...) and the packed tile `tile`.  A row is
// ni floats at memory (i0, k0+k, j0+j); rows that follow each other in memory (a tile as wide as the box) move as one block.
// A 2-D array is the box with nk = nk_m = 1, k0 = 0.
static void tile_rows(float* tile, float* mem, const kidmp_wrf_tile& t, long ni_m, long nk_m, bool to_tile) {
  long run = t.ni;
  int nkr = t.nk, njr = t.nj;
  if (t.ni == ni_m) { run *= t.nk; nkr = 1; if (t.nk == nk_m) { run *= t.nj; njr = 1; } }
  for (int j = 0; j < njr; ++j)
    for (int k = 0; k < nkr; ++k) {
      float* const m = mem + t.i0 + ni_m * (t.k0 + k + nk_m * (long)(t.j0 + j));
      float* const p = tile + ((long)k + (long)t.nk * j) * t.ni;
      if (to_tile) memcpy(p, m, run * 4); else memcpy(m, p, run * 4);
    }
}

int kidmp_mp_gt_driver_tile(kidmp_handle* h, const kidmp_wrf_fields* w, const kidmp_wrf_tile* t, const kidmp_wrf_aerosols* ae,
                            float dt_in) {
  if (!h) return 1;
  if (h->multi) return kidmp_mp_gt_driver_tile(h->multi->dev[0], w, t, ae, dt_in) ? fail(h, "%s", h->multi->dev[0]->err.c_str()) : 0;   // one tile, one device
  if (wrf_check(h, ae ? "mp_gt_driver_aero" : "mp_gt_driver", w, t, ae, dt_in)) return 1;
  const bool radii = w->re_cloud && w->re_ice && w->re_snow;
  const long ncol = (long)t->ni * t->nj;
  if (kidmp_state_alloc(h, ncol, t->nk)) return 1;
  DevGuard guard_(h->device);
  const size_t n = (size_t)ncol * t->nk, n2 = (size_t)ncol;
  // device staging: 12 three-dimensional inputs, the per-column dz in step layout, 3 radii, 7 two-dimensional arrays
  if (ensure_dev(h, &h->d_kid, &h->kid_floats, (12 + 1 + 3) * n + 7 * n2)) return 1;
  // one pinned buffer, one copy each way (as kidmp_kid_interface): the tile of the 12 inputs, 7 accumulators, 4 aerosol arrays + nwfa2d
  const size_t hfloats = 12 * n + 7 * n2 + (ae ? 4 * n + n2 : 0);
  if (h->h_kid_floats < hfloats) {
    if (h->h_kid) cudaFreeHost(h->h_kid);
    h->h_kid = nullptr; h->h_kid_floats = 0;
    CK(h, cudaHostAlloc((void**)&h->h_kid, hfloats * 4, cudaHostAllocDefault));
    h->h_kid_floats = hfloats;
  }
  // aerosol-aware: planes (4 n + n2) for wrf_kernels, then the packed tile of the 4 arrays and nwfa2d
  if (ae && ensure_dev(h, &h->d_aero, &h->aero_floats, 2 * (4 * n + n2))) return 1;
  const long ni_m = w->ni, nk_m = w->nk;
  const kidmp_wrf_tile t2{t->i0, t->ni, 0, 1, t->j0, t->nj};
  CK(h, cudaStreamWaitEvent(h->stream, h->ev_done, 0));  // (the device staging may still serve a call on another stream)
  float* const io[9] = {w->qv, w->qc, w->qi, w->qr, w->qs, w->qg, w->ni_, w->nr, w->th};      // state-field order
  const float* const in3[12] = {w->qv, w->qc, w->qi, w->qr, w->qs, w->qg, w->ni_, w->nr, w->th, w->pii, w->p, w->dz};
  for (int q = 0; q < 12; ++q) tile_rows(h->h_kid + n * q, const_cast<float*>(in3[q]), *t, ni_m, nk_m, true);   // (read only)
  float* const h_2d = h->h_kid + n * 12;
  float* const acc[7] = {w->rainnc, w->rainncv, w->sr, w->snownc, w->snowncv, w->graupelnc, w->graupelncv};
  for (int q = 0; q < 7; ++q) if (acc[q]) tile_rows(h_2d + n2 * q, acc[q], t2, ni_m, 1, true);
  float* const h_ae = h_2d + 7 * n2;
  if (ae) {
    const float* const in4[4] = {ae->nc, ae->nwfa, ae->nifa, ae->w};
    for (int q = 0; q < 4; ++q) tile_rows(h_ae + n * q, const_cast<float*>(in4[q]), *t, ni_m, nk_m, true);
    if (ae->nwfa2d) tile_rows(h_ae + 4 * n, const_cast<float*>(ae->nwfa2d), t2, ni_m, 1, true);
  }
  // on the device the packed tile is a memory box of its own
  WrfArgs a{};
  a.t = WrfBox{t->ni, t->nk, t->nj, 0, 0, 0, t->ni, t->nk};
  for (int q = 0; q < 9; ++q) a.a3[q] = h->d_kid + n * q;
  a.pii = h->d_kid + n * 9; a.p3 = h->d_kid + n * 10; a.dz3 = h->d_kid + n * 11;
  a.dz_col = h->d_kid + n * 12;
  float* const d_re = h->d_kid + n * 13;
  if (radii) { a.re_cloud = d_re; a.re_ice = d_re + n; a.re_snow = d_re + 2 * n; }
  float* const d_2d = h->d_kid + n * 16;
  a.rainnc = d_2d; a.rainncv = d_2d + n2; a.sr = d_2d + 2 * n2;
  if (w->snownc && w->snowncv) { a.snownc = d_2d + 3 * n2; a.snowncv = d_2d + 4 * n2; }
  if (w->graupelnc && w->graupelncv) { a.graupelnc = d_2d + 5 * n2; a.graupelncv = d_2d + 6 * n2; }
  float* const d_aet = ae ? h->d_aero + 4 * n + n2 : nullptr;
  CK(h, cudaMemcpyAsync(h->d_kid, h->h_kid, 12 * n * 4, cudaMemcpyHostToDevice, h->stream));
  CK(h, cudaMemcpyAsync(d_2d, h_2d, 7 * n2 * 4, cudaMemcpyHostToDevice, h->stream));
  if (ae) CK(h, cudaMemcpyAsync(d_aet, h_ae, (4 * n + n2) * 4, cudaMemcpyHostToDevice, h->stream));
  float* const ae4[4] = {d_aet, d_aet + n, d_aet + 2 * n, d_aet + 3 * n};
  if (wrf_kernels(h, a, ae ? ae4 : nullptr, ae && ae->nwfa2d ? d_aet + 4 * n : nullptr, dt_in, h->stream)) return 1;
  CK(h, cudaMemcpyAsync(h->h_kid, h->d_kid, 9 * n * 4, cudaMemcpyDeviceToHost, h->stream));
  float* const h_re = h->h_kid + n * 9;               // pii, p, dz slots of the pinned buffer are free again
  if (radii) CK(h, cudaMemcpyAsync(h_re, d_re, 3 * n * 4, cudaMemcpyDeviceToHost, h->stream));
  CK(h, cudaMemcpyAsync(h_2d, d_2d, 7 * n2 * 4, cudaMemcpyDeviceToHost, h->stream));
  if (ae) CK(h, cudaMemcpyAsync(h_ae, d_aet, 3 * n * 4, cudaMemcpyDeviceToHost, h->stream));
  CK(h, cudaStreamSynchronize(h->stream));
  for (int q = 0; q < 9; ++q) tile_rows(h->h_kid + n * q, io[q], *t, ni_m, nk_m, false);
  if (radii) {
    float* const re[3] = {w->re_cloud, w->re_ice, w->re_snow};
    for (int q = 0; q < 3; ++q) tile_rows(h_re + n * q, re[q], *t, ni_m, nk_m, false);
  }
  for (int q = 0; q < 3; ++q) tile_rows(h_2d + n2 * q, acc[q], t2, ni_m, 1, false);
  if (a.snownc) for (int q = 3; q < 5; ++q) tile_rows(h_2d + n2 * q, acc[q], t2, ni_m, 1, false);
  if (a.graupelnc) for (int q = 5; q < 7; ++q) tile_rows(h_2d + n2 * q, acc[q], t2, ni_m, 1, false);
  if (ae) {
    float* const out3[3] = {ae->nc, ae->nwfa, ae->nifa};
    for (int q = 0; q < 3; ++q) tile_rows(h_ae + n * q, out3[q], *t, ni_m, nk_m, false);
  }
  return 0;
}

int kidmp_mp_gt_driver_tile_device(kidmp_handle* h, const kidmp_wrf_fields* w, const kidmp_wrf_tile* t,
                                   const kidmp_wrf_aerosols* ae, float dt_in, void* stream) {
  if (!h) return 1;
  if (h->multi) return fail(h, "mp_gt_driver_tile_device: device pointers belong to one device; use a single-device handle per GPU");
  if (wrf_check(h, "mp_gt_driver_tile_device", w, t, ae, dt_in)) return 1;
  const long ncol = (long)t->ni * t->nj;
  if (kidmp_state_alloc(h, ncol, t->nk)) return 1;
  DevGuard guard_(h->device);
  const size_t n = (size_t)ncol * t->nk, n2 = (size_t)ncol;
  if (ensure_dev(h, &h->d_kid, &h->kid_floats, n)) return 1;          // the per-column dz in step layout
  if (ae && ensure_dev(h, &h->d_aero, &h->aero_floats, 4 * n + n2)) return 1;
  WrfArgs a{};
  a.t = WrfBox{t->ni, t->nk, t->nj, t->i0, t->k0, t->j0, w->ni, w->nk};
  float* const io[9] = {w->qv, w->qc, w->qi, w->qr, w->qs, w->qg, w->ni_, w->nr, w->th};
  for (int q = 0; q < 9; ++q) a.a3[q] = io[q];
  a.pii = w->pii; a.p3 = w->p; a.dz3 = w->dz;
  a.dz_col = h->d_kid;
  if (w->re_cloud && w->re_ice && w->re_snow) { a.re_cloud = w->re_cloud; a.re_ice = w->re_ice; a.re_snow = w->re_snow; }
  a.rainnc = w->rainnc; a.rainncv = w->rainncv; a.sr = w->sr;
  if (w->snownc && w->snowncv) { a.snownc = w->snownc; a.snowncv = w->snowncv; }
  if (w->graupelnc && w->graupelncv) { a.graupelnc = w->graupelnc; a.graupelncv = w->graupelncv; }
  cudaStream_t s = stream ? (cudaStream_t)stream : h->stream;
  float* const ae4[4] = {ae ? ae->nc : nullptr, ae ? ae->nwfa : nullptr, ae ? ae->nifa : nullptr, ae ? const_cast<float*>(ae->w) : nullptr};
  return wrf_kernels(h, a, ae ? ae4 : nullptr, ae ? ae->nwfa2d : nullptr, dt_in, s);
}

int kidmp_set_option(kidmp_handle* h, const char* name, int value) {
  if (!h) return 1;
  if (h->multi) {
    for (kidmp_handle* c : h->multi->dev) if (kidmp_set_option(c, name, value)) return fail(h, "%s", c->err.c_str());
    return 0;
  }
  if (!name) return fail(h, "set_option: null name");
  if (!strcmp(name, "chunk")) {
    if (value < 32) return fail(h, "set_option: chunk must be at least 32 columns");
    h->chunk_cols = value; return 0;
  }
  if (!strcmp(name, "graphs")) { h->graphs = value != 0; return 0; }
  if (!strcmp(name, "simple")) { h->simple = value != 0; return 0; }
  if (!strcmp(name, "classes")) { h->classes = value != 0; return 0; }
  if (!strcmp(name, "timing")) { h->timing = value < 0 ? 0 : value > 2 ? 2 : value; h->timing_valid = false; return 0; }
  return fail(h, "set_option: unknown option '%s'", name);
}

long kidmp_gpu_launches(const kidmp_handle* h) {
  if (h && h->multi) { long n = 0; for (kidmp_handle* c : h->multi->dev) n += c->launches; return n; }
  return h ? h->launches : 0;
}

const char* kidmp_kernel_names(void) {
  return "classify,lists,n0_sweep,cells_warm,cells_ice,cells_mixed_no_rain,cells_full,carries,substeps,finish,diag";
}

int kidmp_last_kernel_ms(kidmp_handle* h, float* out, int n) {
  if (!h || !out) return 1;
  if (h->multi) return kidmp_last_kernel_ms(h->multi->dev[0], out, n);
  if (!h->timing_valid) return fail(h, "last_kernel_ms: set_option(\"timing\", 1) before the step");
  DevGuard guard_(h->device);
  CK(h, cudaEventSynchronize(h->ev_k[KT_N]));
  for (int q = 0; q < n && q < KT_N; ++q) CK(h, cudaEventElapsedTime(out + q, h->ev_k[q], h->ev_k[q + 1]));
  return 0;
}

int kidmp_step_stats(kidmp_handle* h, long out[8]) {
  if (!h || !out) return 1;
  if (h->multi) {                                       // summed over the devices
    for (int q = 0; q < 8; ++q) out[q] = 0;
    for (kidmp_handle* c : h->multi->dev) {
      long one[8];
      if (kidmp_step_stats(c, one)) return fail(h, "%s", c->err.c_str());
      for (int q = 0; q < 8; ++q) out[q] += one[q];
    }
    return 0;
  }
  for (int q = 0; q < 8; ++q) out[q] = 0;
  DevGuard guard_(h->device);
  CK(h, cudaEventSynchronize(h->ev_done));
  if (h->ws.d_cellmeta) {                               // the last launch of the last step
    int meta[8], cloudy = 0;
    CK(h, cudaMemcpy(meta, h->ws.d_cellmeta, sizeof meta, cudaMemcpyDeviceToHost));
    CK(h, cudaMemcpy(&cloudy, h->ws.d_work, 4, cudaMemcpyDeviceToHost));
    out[0] = cloudy; out[1] = meta[KC_N];
    for (int q = 0; q < KC_N; ++q) out[2 + q] = meta[q];
    out[6] = meta[5];
  }
  out[7] = h->last_zero_copy ? 1 : 0;
  return 0;
}

int kidmp_sync(kidmp_handle* h) {
  if (!h) return 1;
  if (h->multi) {
    for (kidmp_handle* c : h->multi->dev) if (kidmp_sync(c)) return fail(h, "%s", c->err.c_str());
    return 0;
  }
  DevGuard guard_(h->device);
  CK(h, cudaStreamSynchronize(h->stream));
  return 0;
}

int kidmp_last_step_ms(kidmp_handle* h, float* step_ms) {
  if (!h || !step_ms) return 1;
  if (h->multi) {                                       // the slowest device
    *step_ms = 0.f;
    for (kidmp_handle* c : h->multi->dev) {
      float ms = 0.f;
      if (kidmp_last_step_ms(c, &ms)) return fail(h, "%s", c->err.c_str());
      if (ms > *step_ms) *step_ms = ms;
    }
    return 0;
  }
  DevGuard guard_(h->device);
  if (!h->last_on_own_stream) return fail(h, "last_step_ms: the last step ran on a caller's stream; time it there");
  CK(h, cudaEventSynchronize(h->ev1));
  CK(h, cudaEventElapsedTime(step_ms, h->ev0, h->ev1));
  return 0;
}

int kidmp_kid_interface(kidmp_handle* h, const kidmp_kid_columns* c, float dt, float p0, float r_on_cp) {
  if (!h) return 1;
  if (!c) return fail(h, "kid_interface: null argument");
  if (c->nx == 0) return 0;                              // an empty domain is not an error (I:54)
  if (h->multi && c->nx >= (long)h->multi->dev.size()) return multi_kid_interface(h, c, dt, p0, r_on_cp);
  if (h->multi) return kidmp_kid_interface(h->multi->dev[0], c, dt, p0, r_on_cp) ? fail(h, "%s", h->multi->dev[0]->err.c_str()) : 0;
  if (!c->theta || !c->dtheta_adv || !c->dtheta_div || !c->exner || !c->qv || !c->dqv_adv || !c->dqv_div || !c->dz ||
      !c->dtheta_mphys || !c->dqv_mphys || !c->ppt)
    return fail(h, "kid_interface: null array");
  const bool warm = h->kc.iiwarm != 0;
  for (int m = 0; m < 7; ++m) {
    const bool need = m < 3 || !warm;
    if (need && (!c->hyd[m] || !c->dhyd_adv[m] || !c->dhyd_div[m] || !c->dhyd_mphys[m]))
      return fail(h, "kid_interface: hydrometeor plane %d is null", m);
  }
  if (!(r_on_cp > 0.f) || !(dt > 0.f)) return fail(h, "kid_interface: dt and r_on_cp must be positive");
  if (kidmp_state_alloc(h, c->nx, c->nz)) return 1;
  DevGuard guard_(h->device);
  const size_t n = (size_t)c->nx * c->nz;
  const int nplanes = 7 + 21 + 9;
  if (h->kid_floats < n * nplanes) {
    if (h->d_kid) cudaFree(h->d_kid);
    h->d_kid = nullptr; h->kid_floats = 0;
    CK(h, cudaMalloc((void**)&h->d_kid, n * nplanes * 4));
    h->kid_floats = n * nplanes;
  }
  // All planes go through ONE pinned staging buffer and one copy each way: KiD calls this every time step with a
  // handful of columns, where forty small cudaMemcpy calls would cost more than the kernels.
  const size_t nin = 28, nout = 9;
  const size_t hfloats = (nin + nout) * n + (size_t)c->nz + (size_t)c->nx * 4;
  if (h->h_kid_floats < hfloats) {
    if (h->h_kid) cudaFreeHost(h->h_kid);
    h->h_kid = nullptr; h->h_kid_floats = 0;
    CK(h, cudaHostAlloc((void**)&h->h_kid, hfloats * 4, cudaHostAllocDefault));
    h->h_kid_floats = hfloats;
  }
  int slot = 0;
  auto in = [&](const float* src) -> const float* {
    const size_t off = n * (size_t)slot++;
    if (!src) return nullptr;
    memcpy(h->h_kid + off, src, n * 4);
    return h->d_kid + off;
  };
  auto out = [&]() { return h->d_kid + n * (size_t)slot++; };
  KidArgs a{};
  a.nx = c->nx; a.nz = c->nz; a.dt = dt; a.p0 = p0; a.ooroc = 1.f / r_on_cp; a.iiwarm = warm ? 1 : 0;
  a.theta = in(c->theta); a.dtheta_adv = in(c->dtheta_adv); a.dtheta_div = in(c->dtheta_div); a.exner = in(c->exner);
  a.qv = in(c->qv); a.dqv_adv = in(c->dqv_adv); a.dqv_div = in(c->dqv_div);
  for (int m = 0; m < 7; ++m) {
    const bool use = m < 3 || !warm;
    a.hyd[m] = in(use ? c->hyd[m] : nullptr); a.dhyd_adv[m] = in(use ? c->dhyd_adv[m] : nullptr);
    a.dhyd_div[m] = in(use ? c->dhyd_div[m] : nullptr);
  }
  float* const d_out0 = h->d_kid + n * nin;
  a.dtheta_mphys = out(); a.dqv_mphys = out();
  for (int m = 0; m < 7; ++m) a.dhyd_mphys[m] = out();
  float* const h_dz = h->h_kid + (nin + nout) * n;
  float* const h_ppt = h_dz + c->nz;
  memcpy(h_dz, c->dz, (size_t)c->nz * 4);
  for (int q = 0; q < KIDMP_NFIELDS; ++q) a.f[q] = field_ptr(h, q);
  a.p = field_ptr(h, KIDMP_NFIELDS);
  CK(h, cudaMemcpyAsync(h->d_kid, h->h_kid, (warm ? (7 + 9) : nin) * n * 4, cudaMemcpyHostToDevice, h->stream));
  CK(h, cudaMemcpyAsync(h->d_dz, h_dz, (size_t)c->nz * 4, cudaMemcpyHostToDevice, h->stream));
  dim3 g((unsigned)((c->nx + 31) / 32), (unsigned)((c->nz + 31) / 32)), b(32, 8);
  k_kid_gather<<<g, b, 0, h->stream>>>(a);
  ++h->launches;
  CK(h, cudaEventRecord(h->ev0, h->stream));
  if (launch_step(h, resident_args(h, dt), h->stream)) return 1;
  CK(h, cudaEventRecord(h->ev1, h->stream));
  k_kid_scatter<<<g, b, 0, h->stream>>>(a);
  ++h->launches;
  CK(h, cudaGetLastError());
  float* const h_out0 = h->h_kid + n * nin;
  CK(h, cudaMemcpyAsync(h_out0, d_out0, (warm ? 5 : nout) * n * 4, cudaMemcpyDeviceToHost, h->stream));
  CK(h, cudaMemcpyAsync(h_ppt, h->d_ppt, (size_t)c->nx * 16, cudaMemcpyDeviceToHost, h->stream));
  CK(h, cudaStreamSynchronize(h->stream));
  memcpy(c->dtheta_mphys, h_out0, n * 4);
  memcpy(c->dqv_mphys, h_out0 + n, n * 4);
  for (int m = 0; m < 7; ++m)
    if (m < 3 || !warm) memcpy(c->dhyd_mphys[m], h_out0 + n * (size_t)(2 + m), n * 4);
  memcpy(c->ppt, h_ppt, (size_t)c->nx * 16);
  return 0;
}

void* kidmp_stream(kidmp_handle* h) { return h && !h->multi ? (void*)h->stream : nullptr; }
int kidmp_num_devices(const kidmp_handle* h) { return !h ? 0 : h->multi ? (int)h->multi->dev.size() : 1; }

int kidmp_device_state(kidmp_handle* h, float* d_fields[KIDMP_NFIELDS], float** d_p, float** d_dz, float** d_ppt) {
  if (h && h->multi) return fail(h, "device_state: device pointers belong to one device; use a single-device handle");
  if (!h || !h->d_state) return h ? fail(h, "device_state before state_alloc") : 1;
  for (int q = 0; q < KIDMP_NFIELDS; ++q) if (d_fields) d_fields[q] = field_ptr(h, q);
  if (d_p) *d_p = field_ptr(h, KIDMP_NFIELDS);
  if (d_dz) *d_dz = h->d_dz;
  if (d_ppt) *d_ppt = h->d_ppt;
  return 0;
}

}  // extern "C"
