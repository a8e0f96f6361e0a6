// C ABI of libeggshell_b200.so (declared in include/egg_cuda.h).  Host-side plumbing only:
// device allocation, AoS<->SoA staging, kernel sequencing for Ensemble::Step
// (/root/reference/eggshell/ensembles.cc:390-427).  There is no CPU fallback: without a CUDA
// device every entry point fails with EGG_ERR_NO_DEVICE.
#include "../../include/egg_cuda.h"
#include "egg_internal.cuh"
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>
#include <algorithm>
#include <climits>
#include <cstdint>
#include <limits>
#include <initializer_list>

cudaError_t egg_launch_solve_dense(const EggDev& d, double dt, cudaStream_t s, void* scratch, size_t scratch_bytes);
size_t egg_dense_scratch_bytes(const EggDev& d);
int egg_dense_smem_fits(const EggDev& d, size_t limit);
double egg_measure_fp64_tflops();
cudaError_t egg_launch_relax(const EggDev& d, double dt, double step_scale, int max_steps, int mode, void* scratch, size_t scratch_bytes,
                             int* prog, double* err2, int* any_active, cudaStream_t s);

static thread_local std::string g_err;
static int env_int(const char* name, int dflt) {
  const char* e = getenv(name);
  return e ? atoi(e) : dflt;
}
static void set_err(const char* what, cudaError_t e) {
  char buf[512];
  snprintf(buf, sizeof(buf), "%s: %s", what, cudaGetErrorString(e));
  g_err = buf;
}
#define CK(call)                                \
  do {                                          \
    cudaError_t e__ = (call);                   \
    if (e__ != cudaSuccess) {                   \
      set_err(#call, e__);                      \
      return EGG_ERR_CUDA;                      \
    }                                           \
  } while (0)
// CK for egg_create after the batch exists: releases it on failure
#define CKB(call)                               \
  do {                                          \
    cudaError_t e__ = (call);                   \
    if (e__ != cudaSuccess) {                   \
      set_err(#call, e__);                      \
      egg_destroy(b);                           \
      return EGG_ERR_CUDA;                      \
    }                                           \
  } while (0)

struct egg_batch {
  egg_desc desc;
  EggDev dev;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  bool initialised = false;
  bool iso_known = false;     // dev.iso read back from the device after egg_init
  std::vector<void*> allocs;
  long long bytes = 0;
  long long launches = 0;
  double* stage = nullptr;        // device staging for AoS <-> SoA conversion
  size_t stage_bytes = 0;
  void* dense_scratch = nullptr;
  size_t dense_scratch_bytes = 0;
  int* relax_prog = nullptr;     // [2 W] relaxation progress, allocated by the first stabilisation call
  double* relax_err2 = nullptr;  // [W]
  int* relax_any = nullptr;      // [1]
  double* rec_aux = nullptr;     // per-world records for the relaxation when dev.rec holds the PGS group stream
  int* level_aux = nullptr;
  int device = 0;
  double* snap = nullptr;        // egg_snapshot copy of dev.dyn
  int* gather_idx = nullptr;     // [W] world indices of egg_gather_state, allocated by its first call
  double* cost_buf = nullptr;    // egg_set_cost arrays (EggCost layout); null = no cost set
  size_t cost_count = 0;
  EggCost cost = {};             // pointers into cost_buf
  double* sampler_buf = nullptr; // egg_set_sampler arrays (EggSampler layout); null = no sampler set
  size_t sampler_count = 0;
  EggSampler sampler = {};       // pointers into sampler_buf
  double* mppi_partial = nullptr;  // stage-1 partials of egg_mppi_reduce, grown on demand
  size_t mppi_partial_count = 0;
  int* act_ibuf = nullptr;       // egg_set_actuators: body, reaction, frame [m], CSR start [n + 1], list; null = body wrenches
  size_t act_icount = 0;
  double* act_dbuf = nullptr;    // ... and axis [m][3]
  size_t act_dcount = 0;
  EggAct act = {};               // pointers into act_ibuf / act_dbuf; act.m = 0 without a table
  double* mu = nullptr;          // egg_set_friction: [W] Coulomb friction coefficients; null = BOX friction
  size_t mu_count = 0;
  bool profiling = false;
  std::vector<cudaEvent_t> ev;   // 4 per profiled step
  std::vector<cudaEvent_t> ev_free;
};

template <class T>
static int dalloc(egg_batch* b, T** p, size_t count) {
  size_t bytes = count * sizeof(T);
  if (bytes == 0) bytes = sizeof(T);
  void* q = nullptr;
  cudaError_t e = cudaMalloc(&q, bytes);
  if (e != cudaSuccess) { set_err("cudaMalloc", e); return EGG_ERR_CUDA; }
  e = cudaMemsetAsync(q, 0, bytes, b->stream);
  if (e != cudaSuccess) { set_err("cudaMemset", e); return EGG_ERR_CUDA; }
  b->allocs.push_back(q);
  b->bytes += (long long)bytes;
  *p = (T*)q;
  return EGG_OK;
}
// Releases one dalloc'd buffer before egg_destroy, once the work queued on the stream is done with it.
static int dfree(egg_batch* b, void* p, size_t bytes) {
  CK(cudaStreamSynchronize(b->stream));
  CK(cudaFree(p));
  b->allocs.erase(std::find(b->allocs.begin(), b->allocs.end(), p));
  b->bytes -= (long long)bytes;
  return EGG_OK;
}
#define RET(x) do { int r__ = (x); if (r__ != EGG_OK) return r__; } while (0)
// Replaces the batch-owned buffer buf of count elements with a new one of new_count elements (none if
// 0), filled from host if given.  The new buffer is in place before the old one goes, so a failed
// allocation keeps the old buffer; the stream is synchronised before the old one is freed.
template <class T>
static int replace_dbuf(egg_batch* b, T*& buf, size_t& count, size_t new_count, const T* host) {
  T* q = nullptr;
  if (new_count) {
    RET(dalloc(b, &q, new_count));
    if (host) CK(cudaMemcpyAsync(q, host, new_count * sizeof(T), cudaMemcpyHostToDevice, b->stream));
  }
  CK(cudaStreamSynchronize(b->stream));   // host may be a temporary
  if (buf) RET(dfree(b, buf, count * sizeof(T)));
  buf = q;
  count = new_count;
  return EGG_OK;
}
#define DA(ptr, count)                                  \
  do {                                                  \
    int r__ = dalloc(b, &(ptr), (size_t)(count));       \
    if (r__ != EGG_OK) { egg_destroy(b); return r__; }  \
  } while (0)

extern "C" {

const char* egg_last_error(void) { return g_err.c_str(); }
const char* egg_version(void) { return "eggshell_b200 0.1 (sm_100a)"; }

int egg_desc_default(egg_desc* d, int n_worlds, int n_bodies, int n_joints) {
  if (!d) return EGG_ERR_ARG;
  memset(d, 0, sizeof(*d));
  d->n_worlds = n_worlds;
  d->n_bodies = n_bodies;
  d->n_joints = n_joints;
  d->max_contacts = 0;
  d->precision = 64;
  d->solver = EGG_SOLVER_DENSE_MURTY;   // what the reference ships (ensembles.cc:21)
  d->k_max = 500;                       // sparse_iterations.cc:19
  d->tol = 1e-9;                        // constants.h:5
  d->cfm = 0.01;                        // ensembles.cc:14
  d->erp = 0.2;                         // ensembles.h:166
  d->gravity[0] = 0; d->gravity[1] = 0; d->gravity[2] = -9.8;   // constants.h:8
  d->min_constraint_dist = 1e-6;        // ensembles.cc:15
  d->quirks = EGG_QUIRKS_REFERENCE;
  d->cfm_mode = EGG_CFM_AUTO;
  d->device = 0;
  d->taps = 0;
  return EGG_OK;
}

int egg_create(const egg_desc* dsc, egg_batch** out) {
  if (!dsc || !out) return EGG_ERR_ARG;
  *out = nullptr;
  if (dsc->n_worlds <= 0 || dsc->n_bodies <= 0 || dsc->n_joints < 0 || dsc->n_bodies > 360) { g_err = "bad shape"; return EGG_ERR_ARG; }
  if (dsc->precision != 64 && dsc->precision != 32) { g_err = "precision must be 64 or 32"; return EGG_ERR_ARG; }
  if (dsc->precision == 32 && dsc->solver != EGG_SOLVER_PGS) { g_err = "precision = 32 (FP32 constraint records) exists for the PGS solver only"; return EGG_ERR_UNSUPPORTED; }
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) {
    g_err = "no CUDA device: eggshell_b200 has no CPU fallback";
    return EGG_ERR_NO_DEVICE;
  }
  if (dsc->device < 0 || dsc->device >= ndev) { g_err = "bad device ordinal"; return EGG_ERR_ARG; }
  CK(cudaSetDevice(dsc->device));
  egg_batch* b = new egg_batch();
  b->desc = *dsc;
  b->device = dsc->device;
  e = cudaStreamCreateWithFlags(&b->stream, cudaStreamNonBlocking);
  if (e != cudaSuccess) { set_err("cudaStreamCreate", e); delete b; return EGG_ERR_CUDA; }
  b->own_stream = true;

  EggDev& d = b->dev;
  memset(&d, 0, sizeof(d));
  const int W = dsc->n_worlds, n = dsc->n_bodies, nj = dsc->n_joints;
  d.W = W; d.n = n; d.nj = nj;
  d.P = n * (n - 1) / 2;
  // Capacity: 8 ground contacts per body is exact (collision.cc:412-414); pairs emit <= 10 each
  // (4-gon clipped by 6 half-spaces).  Automatic = 8 n + 4 contacts for ~4 colliding pairs/body.
  int maxc = dsc->max_contacts > 0 ? dsc->max_contacts : 8 * n + 16 * n;
  if (maxc > 8 * n + 10 * d.P) maxc = 8 * n + 10 * d.P;
  if (maxc < 8) maxc = 8;
  maxc = (maxc + 7) & ~7;
  d.maxc = maxc;
  d.nrec = nj + maxc;
  b->desc.max_contacts = maxc;
  d.prm.erp = dsc->erp; d.prm.cfm = dsc->cfm; d.prm.tol = dsc->tol; d.prm.min_dist = dsc->min_constraint_dist;
  for (int k = 0; k < 3; k++) d.prm.g[k] = dsc->gravity[k];
  d.prm.k_max = dsc->k_max; d.prm.solver = dsc->solver; d.prm.quirks = dsc->quirks; d.prm.cfm_mode = dsc->cfm_mode;
  // kernel-selection overrides: read here, once per batch (egg_get_kernel_config reports the result)
  d.sel.lpw = env_int("EGG_PGS_LPW", 0);
  d.sel.min_warps = env_int("EGG_PGS_MIN_WARPS_PER_SM", 3);
  d.sel.runs = getenv("EGG_PGS_RUNS") ? (env_int("EGG_PGS_RUNS", 0) != 0) : -1;
  d.sel.run_cap = env_int("EGG_PGS_RUN_CAP", 0);
  d.sel.target_ctas = env_int("EGG_PGS_TARGET_CTAS", 11);
  if (d.sel.target_ctas < 1) d.sel.target_ctas = 11;
  d.sel.collide_nt = env_int("EGG_COLLIDE_NT", 0);
  d.sel.records_nt = env_int("EGG_RECORDS_NT", 0);
  d.sel.ctas_per_sm = env_int("EGG_PGS_CTAS_PER_SM", 0);
  d.sel.pf = env_int("EGG_PGS_PF", 3);

  DA(d.dyn, (size_t)W * EGG_DYN * n);
  DA(d.stat, (size_t)W * EGG_STAT * n);
  DA(d.bpar, (size_t)W * EGG_BPAR * n);
  DA(d.minv_aos, (size_t)W * (n + 1) * 10);
  DA(d.j_i0, (size_t)W * nj);
  DA(d.j_i1, (size_t)W * nj);
  DA(d.jc, (size_t)W * 6 * nj);
  DA(d.c_count, W);
  DA(d.c_i0, (size_t)W * maxc);
  DA(d.c_i1, (size_t)W * maxc);
  DA(d.c_code, (size_t)W * maxc);
  DA(d.c_geom, (size_t)W * 7 * maxc);
  if (dsc->taps) {
    DA(d.pair_code, (size_t)W * d.P);
    DA(d.pair_cnt, (size_t)W * d.P);
  }
  // The PGS solver streams group-interleaved records (format 1, egg_pgs_stream.cu); the dense path,
  // Jacobi / SOR and the relaxation read per-world 240-byte records (format 0, egg_pgs.cu).
  d.rec_fmt = (dsc->solver == EGG_SOLVER_PGS) ? 1 : 0;
  d.rmax = 0;
  // the group-stream assembly keeps u16 level tables of 2 (n + 4 nrec) bytes per world in shared memory
  if (d.rec_fmt && d.nrec > 24000) { g_err = "PGS: more than 24000 constraint slots per world (n_joints + max_contacts) are not supported"; egg_destroy(b); return EGG_ERR_UNSUPPORTED; }
  if (d.rec_fmt) {
    // group stream: G = 32 / lpw worlds share one interleaved record stream
    d.lpw = egg_stage_cap(d);
    d.blkb = egg_stream_blkb(dsc->precision);
    const int groups = (W + 32 / d.lpw - 1) / (32 / d.lpw);
    DA(d.rec, egg_stream_rec_bytes(W, d.nrec, d.lpw) / sizeof(double));
    DA(d.c_pos, (size_t)W * d.nrec);
    DA(d.st_cnt, (size_t)W * d.nrec);
    // run format (egg_pgs_runs.cu): FP64 records, at most 8 lanes per world; whether the bodies are
    // isotropic (its other condition) is known after egg_init, so the choice is made at the first step
    const bool runs_asked = (dsc->quirks & EGG_OPT_PGS_RUNS) != 0 || d.sel.runs == 1;
    if (runs_asked && dsc->precision == 64 && d.lpw <= 8) {   // [W][nrec] words: only for batches that asked for the run format
      DA(d.st_runs, (size_t)W * d.nrec);
      d.run_cap = egg_run_cap(d);
    }
    DA(d.round_off, (size_t)groups * (d.nrec + 1));
    DA(d.grp_info, (size_t)groups * 4);
  } else {
    DA(d.rec, (size_t)W * d.nrec * EGG_REC);
  }
  if (dsc->solver == EGG_SOLVER_JACOBI || dsc->solver == EGG_SOLVER_SOR) {
    DA(d.lam, (size_t)W * d.nrec * 3);
    DA(d.lam2, (size_t)W * d.nrec * 3);
    DA(d.slot_of, (size_t)W * d.nrec);
  }
  DA(d.lam_out, (size_t)W * d.nrec * 3);
  DA(d.row_state, (size_t)W * d.nrec * 3);
  DA(d.n_levels, W);
  DA(d.status, W);
  DA(d.stats, (size_t)W * 8);
  DA(d.resid, W);
  DA(d.cost0, (size_t)W * 2);
  DA(d.work_ctr, 4);
  DA(d.dbg, 32);
  DA(d.minv_iso, (size_t)W * (n + 1) * 2);
  DA(d.iso_flag, 1);
  b->stage_bytes = (size_t)W * n * 9 * sizeof(double);
  size_t jb = (size_t)W * (nj > 0 ? nj : 1) * 3 * sizeof(double);
  if (jb > b->stage_bytes) b->stage_bytes = jb;
  {   // the contact taps are transposed through the same buffer: room for the geometry of up to 256 worlds at a time
    const size_t cb = (size_t)(W < 256 ? W : 256) * maxc * 3 * sizeof(double);
    if (cb > b->stage_bytes) b->stage_bytes = cb;
  }
  DA(b->stage, b->stage_bytes / sizeof(double));
  // Shared-memory needs of every kernel this batch can launch, against the device limit: an
  // unsupported shape fails here, not as a launch error inside the first egg_step.
  {
    int lim = 0;
    CKB(cudaDeviceGetAttribute(&lim, cudaDevAttrMaxSharedMemoryPerBlockOptin, dsc->device));
    struct { const char* what; size_t need; } req[4] = {
        {"narrowphase (egg_collide_kernel)", egg_collide_smem(d)},
        {"row assembly", d.rec_fmt ? (size_t)0 : egg_assemble_smem(d)},
        {"PGS group stream", d.rec_fmt ? (d.st_runs ? std::max(egg_stream_smem(d), egg_runs_smem(d)) : egg_stream_smem(d)) : (size_t)0},
        {"Jacobi / SOR", (dsc->solver == EGG_SOLVER_JACOBI || dsc->solver == EGG_SOLVER_SOR) ? egg_iter_smem(d) : (size_t)0}};
    for (auto& r : req)
      if (r.need > (size_t)lim) {
        char buf[256];
        snprintf(buf, sizeof(buf), "%s needs %zu bytes of shared memory per CTA for n_bodies = %d, max_contacts = %d; the device offers %d", r.what, r.need, n, maxc, lim);
        g_err = buf;
        egg_destroy(b);
        return EGG_ERR_UNSUPPORTED;
      }
    if (dsc->solver == EGG_SOLVER_DENSE_MURTY && !egg_dense_smem_fits(d, (size_t)lim)) {
      g_err = "dense solver: the row capacity (EGG_DENSE_ROWS / n_joints + 4 n_bodies constraints) does not fit the shared memory of one CTA";
      egg_destroy(b);
      return EGG_ERR_UNSUPPORTED;
    }
  }
  if (dsc->solver == EGG_SOLVER_DENSE_MURTY) {
    DA(d.work, W);
    b->dense_scratch_bytes = egg_dense_scratch_bytes(d);
    char* p = nullptr;
    DA(p, b->dense_scratch_bytes);
    b->dense_scratch = p;
  }
  CKB(cudaStreamSynchronize(b->stream));
  *out = b;
  return EGG_OK;
}

void egg_destroy(egg_batch* b) {
  if (!b) return;
  cudaSetDevice(b->device);
  if (b->stream) cudaStreamSynchronize(b->stream);
  for (void* p : b->allocs) cudaFree(p);
  for (cudaEvent_t e : b->ev) cudaEventDestroy(e);
  for (cudaEvent_t e : b->ev_free) cudaEventDestroy(e);
  if (b->own_stream && b->stream) cudaStreamDestroy(b->stream);
  delete b;
}

int egg_set_stream(egg_batch* b, void* cuda_stream) {
  if (!b) return EGG_ERR_ARG;
  CK(cudaSetDevice(b->device));
  CK(cudaStreamSynchronize(b->stream));
  if (b->own_stream && b->stream) cudaStreamDestroy(b->stream);
  b->stream = (cudaStream_t)cuda_stream;
  b->own_stream = false;
  return EGG_OK;
}

int egg_sync(egg_batch* b) {
  if (!b) return EGG_ERR_ARG;
  CK(cudaSetDevice(b->device));
  CK(cudaStreamSynchronize(b->stream));
  CK(cudaGetLastError());
  return EGG_OK;
}

int egg_set_profiling(egg_batch* b, int on) {
  if (!b) return EGG_ERR_ARG;
  b->profiling = on != 0;
  return EGG_OK;
}
int egg_get_kernel_ms(egg_batch* b, double* out4) {
  if (!b || !out4) return EGG_ERR_ARG;
  CK(cudaSetDevice(b->device));
  CK(cudaStreamSynchronize(b->stream));
  for (int k = 0; k < 4; k++) out4[k] = 0;
  for (size_t s = 0; s + 3 < b->ev.size(); s += 4) {
    for (int k = 0; k < 3; k++) {
      float ms = 0;
      CK(cudaEventElapsedTime(&ms, b->ev[s + k], b->ev[s + k + 1]));
      out4[k] += ms;
    }
    out4[3] += 1;
  }
  for (cudaEvent_t e : b->ev) b->ev_free.push_back(e);
  b->ev.clear();
  return EGG_OK;
}
double egg_fp64_peak_tflops(int device) {
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { g_err = "no CUDA device"; return (double)EGG_ERR_NO_DEVICE; }
  if (cudaSetDevice(device) != cudaSuccess) return (double)EGG_ERR_ARG;
  return egg_measure_fp64_tflops();
}
int egg_get_kernel_config(const egg_batch* b, int out[8]) {
  if (!b || !out) return EGG_ERR_ARG;
  const EggDev& d = b->dev;
  const bool pgs = b->desc.solver == EGG_SOLVER_PGS;
  out[0] = d.lpw;                                          // 0 without the group stream
  out[1] = d.lpw ? 32 / d.lpw : 0;
  out[2] = b->iso_known ? d.iso : -1;
  out[3] = !pgs ? 0 : (!b->iso_known ? -1 : (d.rmax > 0 ? 2 : 1));
  out[4] = (b->iso_known && d.rmax > 0) ? d.run_cap : 0;
  out[5] = b->desc.precision;
  out[6] = egg_collide_threads(d);
  out[7] = egg_assemble_threads(d);
  return EGG_OK;
}
int egg_capacity(const egg_batch* b) { return b ? b->dev.maxc : 0; }
long long egg_device_bytes(const egg_batch* b) { return b ? b->bytes : 0; }
long long egg_launch_count(const egg_batch* b) { return b ? b->launches : 0; }

void* egg_host_alloc(long long bytes) {
  void* p = nullptr;
  if (cudaHostAlloc(&p, (size_t)bytes, cudaHostAllocDefault) != cudaSuccess) return nullptr;
  return p;
}
void egg_host_free(void* p) { if (p) cudaFreeHost(p); }

// Host AoS [W][per_world][comps] -> device SoA component block.
static int upload(egg_batch* b, const double* host, int per_world, int comps, double* soa, int soa_comps, int comp_off) {
  size_t bytes = (size_t)b->dev.W * per_world * comps * sizeof(double);
  if (bytes == 0) return EGG_OK;
  CK(cudaMemcpyAsync(b->stage, host, bytes, cudaMemcpyHostToDevice, b->stream));
  CK(egg_launch_pack(b->dev.W, b->stage, per_world, comps, soa, soa_comps, comp_off, b->stream));
  b->launches++;
  return EGG_OK;
}
static int download(egg_batch* b, double* host, int per_world, int comps, const double* soa, int soa_comps, int comp_off) {
  size_t bytes = (size_t)b->dev.W * per_world * comps * sizeof(double);
  if (bytes == 0) return EGG_OK;
  CK(egg_launch_unpack(b->dev.W, b->stage, per_world, comps, soa, soa_comps, comp_off, b->stream));
  b->launches++;
  CK(cudaMemcpyAsync(host, b->stage, bytes, cudaMemcpyDeviceToHost, b->stream));
  // the staging buffer is reused by the next call
  CK(cudaStreamSynchronize(b->stream));
  return EGG_OK;
}

int egg_set_state(egg_batch* b, const double* p, const double* R, const double* v, const double* w) {
  if (!b) return EGG_ERR_ARG;
  CK(cudaSetDevice(b->device));
  const int n = b->dev.n;
  if (p) RET(upload(b, p, n, 3, b->dev.dyn, EGG_DYN, 0));
  if (R) RET(upload(b, R, n, 9, b->dev.dyn, EGG_DYN, 3));
  if (v) RET(upload(b, v, n, 3, b->dev.dyn, EGG_DYN, 12));
  if (w) RET(upload(b, w, n, 3, b->dev.dyn, EGG_DYN, 15));
  return EGG_OK;
}

int egg_set_bodies(egg_batch* b, const double* p, const double* R, const double* v, const double* w,
                   const double* m, const double* I_body, const double* side) {
  if (!b || !p || !R || !v || !w || !m || !I_body) return EGG_ERR_ARG;
  RET(egg_set_state(b, p, R, v, w));
  const int n = b->dev.n;
  if (side) RET(upload(b, side, n, 3, b->dev.bpar, EGG_BPAR, 0));
  else {
    std::vector<double> s((size_t)b->dev.W * n * 3, 0.3);    // body.h:91
    RET(upload(b, s.data(), n, 3, b->dev.bpar, EGG_BPAR, 0));
    CK(cudaStreamSynchronize(b->stream));
  }
  RET(upload(b, m, n, 1, b->dev.bpar, EGG_BPAR, 3));
  RET(upload(b, I_body, n, 9, b->dev.bpar, EGG_BPAR, 4));
  b->initialised = false;
  return EGG_OK;
}

int egg_set_shapes(egg_batch* b, const int* shape, const double* dims) {
  if (!b || !shape || !dims) return EGG_ERR_ARG;
  CK(cudaSetDevice(b->device));
  const size_t cnt = (size_t)b->dev.W * b->dev.n;
  std::vector<double> t(cnt);
  for (size_t k = 0; k < cnt; k++) {
    if (shape[k] < 0 || shape[k] > 2) { g_err = "collider shape must be 0 (box), 1 (sphere) or 2 (capsule)"; return EGG_ERR_ARG; }
    t[k] = (double)shape[k];
  }
  RET(upload(b, t.data(), b->dev.n, 1, b->dev.bpar, EGG_BPAR, 13));
  CK(cudaStreamSynchronize(b->stream));      // t is a temporary
  RET(upload(b, dims, b->dev.n, 3, b->dev.bpar, EGG_BPAR, 0));
  return EGG_OK;
}

int egg_set_joints(egg_batch* b, const int* i0, const int* i1, const double* c0, const double* c1) {
  if (!b) return EGG_ERR_ARG;
  const int nj = b->dev.nj;
  if (nj == 0) return EGG_OK;
  if (!i0 || !i1 || !c0 || !c1) return EGG_ERR_ARG;
  CK(cudaSetDevice(b->device));
  const size_t cnt = (size_t)b->dev.W * nj;
  for (size_t k = 0; k < cnt; k++) {
    if (i0[k] < 0 || i0[k] >= b->dev.n || i1[k] < -1 || i1[k] >= b->dev.n) { g_err = "joint body index out of range"; return EGG_ERR_ARG; }
  }
  CK(cudaMemcpyAsync(b->dev.j_i0, i0, cnt * sizeof(int), cudaMemcpyHostToDevice, b->stream));
  CK(cudaMemcpyAsync(b->dev.j_i1, i1, cnt * sizeof(int), cudaMemcpyHostToDevice, b->stream));
  RET(upload(b, c0, nj, 3, b->dev.jc, 6, 0));
  RET(upload(b, c1, nj, 3, b->dev.jc, 6, 3));
  b->initialised = false;
  return EGG_OK;
}

int egg_set_external(egg_batch* b, const double* f_ext) {
  if (!b || !f_ext) return EGG_ERR_ARG;
  if (!b->initialised) { g_err = "egg_set_external must follow egg_init"; return EGG_ERR_STATE; }
  CK(cudaSetDevice(b->device));
  return upload(b, f_ext, b->dev.n, 6, b->dev.stat, EGG_STAT, 10);
}

int egg_init(egg_batch* b) {
  if (!b) return EGG_ERR_ARG;
  CK(cudaSetDevice(b->device));
  CK(egg_launch_init(b->dev, b->stream));
  b->launches += (b->dev.nj > 0) ? 3 : 2;
  // Ensemble::Init ends with CheckAndCorrectEnsembleState (ensembles.cc:28): the joint-joint
  // conflict scan lives in the narrowphase kernel, so run it once here -- EGG_ST_JOINT_CONFLICT is
  // then visible right after egg_init, as the reference's Panic would be.
  CK(egg_launch_collide(b->dev, b->stream));
  CK(egg_launch_clear_contacts(b->dev, b->stream));   // the contact list stays empty until the first Step / UpdateContacts, as in the reference
  b->launches += 2;
  b->initialised = true;
  b->iso_known = false;
  return EGG_OK;
}

// Shared by egg_init_stabilize / egg_post_stabilize: scratch and progress buffers, allocated once.
static int relax_prepare(egg_batch* b) {
  const int W = b->dev.W;
  if (!b->dense_scratch) {
    if (!egg_dense_smem_fits(b->dev, 227 * 1024)) { g_err = "stabilisation: the row capacity does not fit the shared memory of one CTA"; return EGG_ERR_UNSUPPORTED; }
    b->dense_scratch_bytes = egg_dense_scratch_bytes(b->dev);
    char* p = nullptr;
    int r = dalloc(b, &p, b->dense_scratch_bytes);
    if (r != EGG_OK) return r;
    b->dense_scratch = p;
  }
  if (!b->relax_prog) {
    int r = dalloc(b, &b->relax_prog, (size_t)2 * W); if (r != EGG_OK) return r;
    r = dalloc(b, &b->relax_err2, (size_t)W); if (r != EGG_OK) return r;
    r = dalloc(b, &b->relax_any, (size_t)1); if (r != EGG_OK) return r;
  }
  CK(cudaMemsetAsync(b->relax_prog, 0, (size_t)2 * W * sizeof(int), b->stream));
  return EGG_OK;
}
static int relax_report(egg_batch* b, int* steps_out, double* err_sq_out) {
  const int W = b->dev.W;
  if (steps_out) {
    std::vector<int> h((size_t)2 * W);
    CK(cudaMemcpyAsync(h.data(), b->relax_prog, h.size() * sizeof(int), cudaMemcpyDeviceToHost, b->stream));
    CK(cudaStreamSynchronize(b->stream));
    for (int w = 0; w < W; w++) steps_out[w] = h[2 * w];
  }
  if (err_sq_out) CK(cudaMemcpyAsync(err_sq_out, b->relax_err2, (size_t)W * sizeof(double), cudaMemcpyDeviceToHost, b->stream));
  CK(cudaStreamSynchronize(b->stream));
  CK(cudaGetLastError());
  return EGG_OK;
}

int egg_init_stabilize(egg_batch* b, int max_steps, int* steps_out, double* err_sq_out) {
  if (!b || max_steps < 0) return EGG_ERR_ARG;
  if (!b->initialised) { g_err = "egg_init_stabilize before egg_init"; return EGG_ERR_STATE; }
  CK(cudaSetDevice(b->device));
  RET(relax_prepare(b));
  EggDev nodedup = b->dev;
  nodedup.prm.min_dist = -1.0;   // UpdateContacts only: the loop of ensembles.cc:610-617 never de-duplicates
  nodedup.rec_fmt = 0;           // the relaxation kernel reads per-world records (dev.rec is large enough for either format)
  nodedup.level_start = nullptr;
  const double dt = 0.001 * 500;   // kSimTimeStep * 500 (ensembles.cc:611)
  for (int it = 0; it <= max_steps; it++) {
    CK(egg_launch_collide(nodedup, b->stream));
    CK(egg_launch_assemble(nodedup, dt, b->stream));
    CK(cudaMemsetAsync(b->relax_any, 0, sizeof(int), b->stream));
    CK(egg_launch_relax(nodedup, dt, 0.2, max_steps, 0, b->dense_scratch, b->dense_scratch_bytes, b->relax_prog, b->relax_err2, b->relax_any, b->stream));
    b->launches += 3;
    int h_any = 0;
    CK(cudaMemcpyAsync(&h_any, b->relax_any, sizeof(int), cudaMemcpyDeviceToHost, b->stream));
    CK(cudaStreamSynchronize(b->stream));
    if (!h_any) break;
  }
  CK(egg_launch_collide(b->dev, b->stream));   // CheckAndCorrectEnsembleState (ensembles.cc:618)
  b->launches++;
  return relax_report(b, steps_out, err_sq_out);
}

int egg_post_stabilize(egg_batch* b, int max_steps, int* steps_out, double* err_sq_out) {
  if (!b || max_steps < 0) return EGG_ERR_ARG;
  if (!b->initialised) { g_err = "egg_post_stabilize before egg_init"; return EGG_ERR_STATE; }
  CK(cudaSetDevice(b->device));
  RET(relax_prepare(b));
  EggDev pw = b->dev;
  pw.rec_fmt = 0;
  pw.level_start = nullptr;
  const double dt = 0.001 * 100;   // kSimTimeStep * 100 (ensembles.cc:634)
  // ensembles.cc:624-645: the contact list is NOT refreshed inside this loop; the rows are rebuilt
  // from the current body state and the stored contact geometry every iteration
  for (int it = 0; it <= max_steps; it++) {
    CK(egg_launch_assemble(pw, dt, b->stream));
    CK(cudaMemsetAsync(b->relax_any, 0, sizeof(int), b->stream));
    CK(egg_launch_relax(pw, dt, 0.2, max_steps, 1, b->dense_scratch, b->dense_scratch_bytes, b->relax_prog, b->relax_err2, b->relax_any, b->stream));
    b->launches += 2;
    int h_any = 0;
    CK(cudaMemcpyAsync(&h_any, b->relax_any, sizeof(int), cudaMemcpyDeviceToHost, b->stream));
    CK(cudaStreamSynchronize(b->stream));
    if (!h_any) break;
  }
  return relax_report(b, steps_out, err_sq_out);
}

static int arg_err(const char* what, const char* name, const char* msg) {
  g_err = std::string(what) + "(" + name + "): " + msg;
  return EGG_ERR_ARG;
}
static int check_initialised(egg_batch* b, const char* what) {
  if (!b->initialised) { g_err = std::string(what) + " before egg_init"; return EGG_ERR_STATE; }
  return EGG_OK;
}

// The argument and call-order checks of egg_step and egg_step_controlled.
static int step_check(egg_batch* b, double dt, int integrator, int n_steps, const char* what) {
  if (!b || n_steps < 0 || !(dt > 0)) return EGG_ERR_ARG;
  RET(check_initialised(b, what));
  if (integrator != EGG_OPEN_DYNAMICS_ENGINE) {
    // ensembles.cc:398-405: EXPLICIT_EULER refuses contacts, IMPLICIT_MIDPOINT panics.
    g_err = "only OPEN_DYNAMICS_ENGINE is supported (as in the reference once contacts exist)";
    return EGG_ERR_UNSUPPORTED;
  }
  return EGG_OK;
}

// Where enter() checks that egg_init has run: before or after the device pointers (each entry point
// keeps the order in which it has always checked them), or not at all.
enum InitCheck { INIT_FIRST, INIT_LAST, INIT_NONE };
struct DevArg { const void* p; const char* name; };

// The prologue of the entry points that take device buffers (what: the entry point's name).  A _d
// argument must be device (or managed) memory of the batch's device: a host pointer would reach a
// kernel as an illegal address.  The length behind the pointer cannot be checked here.  align16: the
// double2 accesses of the sampler need 16-byte aligned schedules.
static int enter(egg_batch* b, const char* what, InitCheck init, std::initializer_list<DevArg> ptrs, bool align16 = false) {
  if (!b) return EGG_ERR_ARG;
  if (init == INIT_FIRST) RET(check_initialised(b, what));
  for (const DevArg& a : ptrs) {
    if (!a.p) return arg_err(what, a.name, "NULL device pointer");
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, a.p) != cudaSuccess) { cudaGetLastError(); return arg_err(what, a.name, "not a CUDA pointer"); }
    if ((at.type != cudaMemoryTypeDevice && at.type != cudaMemoryTypeManaged) || at.device != b->device)
      return arg_err(what, a.name, "the buffer is not device memory of the batch's device");
  }
  if (align16)
    for (const DevArg& a : ptrs)
      if ((uintptr_t)a.p & 15) return arg_err(what, a.name, "must be 16-byte aligned");
  if (init == INIT_LAST) RET(check_initialised(b, what));
  CK(cudaSetDevice(b->device));
  return EGG_OK;
}

// The width of a control row per world: m actuator values with an actuator table, else 6 n.
static int ctrl_width(const egg_batch* b) { return b->act.m ? b->act.m : 6 * b->dev.n; }

// n_steps x Ensemble::Step.  With a control schedule u_d ([n_steps][W][c]), slice s is copied into
// the f_ext slot before step s (outside the profiled kernel buckets); with an actuator table the
// actuation kernel writes the slot from the actuator values instead.  With cost_d as well, that
// kernel also adds the running cost of step s to cost_d, and the terminal cost follows the last step.
static int step_loop(egg_batch* b, double dt, int n_steps, const double* u_d, double* cost_d) {
  const int solver = b->dev.prm.solver;
  if (solver < EGG_SOLVER_DENSE_MURTY || solver > EGG_SOLVER_SOR) { g_err = "unknown solver"; return EGG_ERR_ARG; }
  CK(cudaSetDevice(b->device));
  if (!b->iso_known) {   // one 4-byte read-back per egg_init: which M^-1 layout the PGS kernel may use
    int flag = 0;
    CK(cudaMemcpyAsync(&flag, b->dev.iso_flag, sizeof(int), cudaMemcpyDeviceToHost, b->stream));
    CK(cudaStreamSynchronize(b->stream));
    b->dev.iso = !(flag & 1) ? 0 : ((flag & 2) ? 2 : 1);   // 0 general, 1 isotropic, 2 isotropic and uniform
    if (getenv("EGG_PGS_ISO") && atoi(getenv("EGG_PGS_ISO")) < b->dev.iso) b->dev.iso = atoi(getenv("EGG_PGS_ISO"));
    b->iso_known = true;
  }
  // run format of the PGS stream for isotropic bodies, else one block per lane and stage; never with a
  // friction table (BOX friction only).  Decided here, per step, so assembly and solve agree.
  b->dev.rmax = b->mu ? 0 : egg_runs_rmax(b->dev);
  const size_t slice = (size_t)b->dev.W * ctrl_width(b);
  for (int s = 0; s < n_steps; s++) {
    if (u_d) {
      if (b->act.m) CK(egg_launch_actuate(b->dev, b->act, u_d + (size_t)s * slice, cost_d ? &b->cost : nullptr, s, cost_d, b->stream));
      else if (cost_d) CK(egg_launch_fext_slice_cost(b->dev, u_d + (size_t)s * slice, b->cost, s, cost_d, b->stream));
      else CK(egg_launch_fext_slice(b->dev, u_d + (size_t)s * slice, b->stream));
      b->launches++;
    }
    cudaEvent_t e[4] = {nullptr, nullptr, nullptr, nullptr};
    if (b->profiling) {
      for (int k = 0; k < 4; k++) {
        if (!b->ev_free.empty()) { e[k] = b->ev_free.back(); b->ev_free.pop_back(); }
        else CK(cudaEventCreate(&e[k]));
        b->ev.push_back(e[k]);
      }
      CK(cudaEventRecord(e[0], b->stream));
    }
    // EGG_SYNC_DEBUG=1: synchronise after every kernel and name the one that failed
    static const bool dbg_sync = getenv("EGG_SYNC_DEBUG") && atoi(getenv("EGG_SYNC_DEBUG")) != 0;
#define DBG_SYNC(what)                                                                       \
  if (dbg_sync) {                                                                            \
    cudaError_t e__ = cudaStreamSynchronize(b->stream);                                      \
    if (e__ != cudaSuccess) { set_err(what, e__); return EGG_ERR_CUDA; }                      \
  }
    CK(egg_launch_collide(b->dev, b->stream));
    DBG_SYNC("egg_collide_kernel")
    if (b->profiling) CK(cudaEventRecord(e[1], b->stream));
    CK(egg_launch_assemble(b->dev, dt, b->stream));
    DBG_SYNC("assembly kernels")
    if (b->profiling) CK(cudaEventRecord(e[2], b->stream));
    if (solver == EGG_SOLVER_PGS) CK(egg_launch_solve_pgs(b->dev, dt, b->mu, b->stream));
    else if (solver == EGG_SOLVER_DENSE_MURTY) CK(egg_launch_solve_dense(b->dev, dt, b->stream, b->dense_scratch, b->dense_scratch_bytes));
    else CK(egg_launch_solve_iter(b->dev, dt, solver, b->stream));
    DBG_SYNC("solve kernel")
#undef DBG_SYNC
    if (b->profiling) CK(cudaEventRecord(e[3], b->stream));
    b->launches += (solver == EGG_SOLVER_PGS && b->dev.rec_fmt) ? 5 : 3;   // collide, assemble (1 or 3 kernels), solve
  }
  if (cost_d) {
    CK(egg_launch_cost_terminal(b->dev, b->cost, n_steps, cost_d, b->stream));
    b->launches++;
  }
  CK(cudaGetLastError());
  return EGG_OK;
}

int egg_step(egg_batch* b, double dt, int integrator, int n_steps) {
  RET(step_check(b, dt, integrator, n_steps, "egg_step"));
  return step_loop(b, dt, n_steps, nullptr, nullptr);
}

int egg_step_controlled(egg_batch* b, double dt, int integrator, const double* u_d, int horizon) {
  if (!b || !u_d) return EGG_ERR_ARG;
  if (horizon < 1) { g_err = "egg_step_controlled: horizon must be >= 1"; return EGG_ERR_ARG; }
  RET(step_check(b, dt, integrator, horizon, "egg_step_controlled"));
  RET(enter(b, "egg_step_controlled", INIT_NONE, {{u_d, "u_d"}}));
  return step_loop(b, dt, horizon, u_d, nullptr);
}

int egg_step_controlled_cost(egg_batch* b, double dt, int integrator, const double* u_d, int horizon, double* cost_d) {
  if (!b || !u_d) return EGG_ERR_ARG;
  if (horizon < 1) { g_err = "egg_step_controlled_cost: horizon must be >= 1"; return EGG_ERR_ARG; }
  RET(step_check(b, dt, integrator, horizon, "egg_step_controlled_cost"));
  RET(enter(b, "egg_step_controlled_cost", INIT_NONE, {{u_d, "u_d"}, {cost_d, "cost_d"}}));
  if (!b->cost_buf) { g_err = "egg_step_controlled_cost without a cost: call egg_set_cost first"; return EGG_ERR_STATE; }
  if (b->cost.ref_steps > 1 && b->cost.ref_steps < horizon + 1) {
    g_err = "egg_step_controlled_cost: the cost's reference has " + std::to_string(b->cost.ref_steps) + " rows, fewer than horizon + 1 = " +
            std::to_string(horizon + 1);
    return EGG_ERR_ARG;
  }
  return step_loop(b, dt, horizon, u_d, cost_d);
}

int egg_set_friction(egg_batch* b, const double* mu) {
  if (!b) return EGG_ERR_ARG;
  if (b->desc.solver != EGG_SOLVER_PGS) {
    g_err = "egg_set_friction: Coulomb friction exists for the PGS solver only (dense, Jacobi and SOR keep BOX friction)";
    return EGG_ERR_UNSUPPORTED;
  }
  const size_t W = (size_t)b->dev.W;
  std::vector<double> h;
  if (mu) {
    h.resize(W);
    for (size_t w = 0; w < W; w++) {
      if (!std::isfinite(mu[w]) || mu[w] < 0) { g_err = "egg_set_friction: every mu must be finite and >= 0"; return EGG_ERR_ARG; }
      h[w] = mu[w] + 0.0;   // -0.0 -> +0.0
    }
  }
  CK(cudaSetDevice(b->device));
  return replace_dbuf(b, b->mu, b->mu_count, h.size(), h.data());
}

// Host [rows][n][comps] -> component-major [rows][comps][n], the layout of EggCost and EggSampler.
// With finite_only, returns false at the first value that is not finite.
static bool to_component_major(const double* src, size_t rows, size_t n, size_t comps, double* dst, bool finite_only = true) {
  for (size_t r = 0; r < rows; r++)
    for (size_t i = 0; i < n; i++)
      for (size_t k = 0; k < comps; k++) {
        const double v = src[(r * n + i) * comps + k];
        if (finite_only && !std::isfinite(v)) return false;
        dst[(r * comps + k) * n + i] = v;
      }
  return true;
}

int egg_set_cost(egg_batch* b, const egg_cost* c) {
  if (!b) return EGG_ERR_ARG;
  const size_t n = (size_t)b->dev.n, nd = (size_t)EGG_DYN * n, cu = (size_t)ctrl_width(b);
  // the EggCost layout: q_run, l_run, q_term, l_term [18][n], u_run [6][n] (or [m] with an actuator table), x_ref [R][18][n]
  std::vector<double> h;
  int R = 1;
  if (c) {
    if (c->x_ref) R = c->ref_steps;
    if (R < 1) { g_err = "egg_set_cost: ref_steps must be >= 1"; return EGG_ERR_ARG; }
    h.assign(4 * nd + cu + (size_t)R * nd, 0.0);
    const bool act = b->act.m > 0;
    struct { const double* src; size_t rows, n, comps, off; } part[6] = {
        {c->q_run, 1, n, EGG_DYN, 0}, {c->l_run, 1, n, EGG_DYN, nd}, {c->q_term, 1, n, EGG_DYN, 2 * nd},
        {c->l_term, 1, n, EGG_DYN, 3 * nd}, {c->u_run, 1, act ? cu : n, act ? 1 : (size_t)6, 4 * nd},
        {c->x_ref, (size_t)R, n, EGG_DYN, 4 * nd + cu}};
    for (auto& p : part)
      if (p.src && !to_component_major(p.src, p.rows, p.n, p.comps, &h[p.off])) {
        g_err = "egg_set_cost: non-finite weight or reference value";
        return EGG_ERR_ARG;
      }
  }
  CK(cudaSetDevice(b->device));
  RET(replace_dbuf(b, b->cost_buf, b->cost_count, h.size(), h.data()));
  const double* q = b->cost_buf;
  b->cost = c ? EggCost{q, q + nd, q + 4 * nd, q + 2 * nd, q + 3 * nd, q + 4 * nd + cu, R} : EggCost{};
  return EGG_OK;
}

int egg_set_sampler(egg_batch* b, const egg_sampler* s) {
  if (!b) return EGG_ERR_ARG;
  const size_t nc = (size_t)ctrl_width(b);
  std::vector<double> h;   // the EggSampler layout: sigma, lo, hi, each one control row [c] as the host gives it
  if (s) {
    if (!s->sigma) { g_err = "egg_set_sampler: sigma is required"; return EGG_ERR_ARG; }
    const double inf = std::numeric_limits<double>::infinity();
    h.assign(3 * nc, inf);   // without bounds: lo = -inf, hi = +inf
    std::fill(h.begin() + nc, h.begin() + 2 * nc, -inf);
    const bool finite = to_component_major(s->sigma, 1, nc, 1, &h[0]);
    if (s->u_lo) std::copy(s->u_lo, s->u_lo + nc, h.begin() + nc);
    if (s->u_hi) std::copy(s->u_hi, s->u_hi + nc, h.begin() + 2 * nc);
    for (size_t k = 0; k < nc; k++) {
      const double lo = h[nc + k], hi = h[2 * nc + k];
      if (!finite || h[k] < 0) { g_err = "egg_set_sampler: sigma must be finite and >= 0"; return EGG_ERR_ARG; }
      if (std::isnan(lo) || std::isnan(hi)) { g_err = "egg_set_sampler: NaN bound"; return EGG_ERR_ARG; }
      if (lo > hi) { g_err = "egg_set_sampler: u_lo > u_hi"; return EGG_ERR_ARG; }
    }
  }
  CK(cudaSetDevice(b->device));
  RET(replace_dbuf(b, b->sampler_buf, b->sampler_count, h.size(), h.data()));
  const double* q = b->sampler_buf;
  b->sampler = s ? EggSampler{q, q + nc, q + 2 * nc} : EggSampler{};
  return EGG_OK;
}

int egg_set_actuators(egg_batch* b, const egg_actuators* a) {
  if (!b) return EGG_ERR_ARG;
  if (b->sampler_buf || b->cost_buf) {
    g_err = "egg_set_actuators while a sampler or a cost is set: their control rows have the width of the current control space; "
            "clear them first";
    return EGG_ERR_STATE;
  }
  const int n = b->dev.n;
  std::vector<int> hi;      // body, reaction, frame [m], start [n + 1], list
  std::vector<double> hd;   // axis [m][3]
  int m = 0;
  if (a) {
    m = a->m;
    if (m < 1 || m > INT_MAX / 8) { g_err = "egg_set_actuators: m must be in [1, INT_MAX / 8]"; return EGG_ERR_ARG; }
    if (!a->body || !a->reaction || !a->frame || !a->axis) { g_err = "egg_set_actuators: NULL array"; return EGG_ERR_ARG; }
    std::vector<int> cnt((size_t)n + 1, 0);
    for (int k = 0; k < m; k++) {
      const int bo = a->body[k], re = a->reaction[k], fr = a->frame[k];
      const double* ax = a->axis + 3 * (size_t)k;
      if (bo < 0 || bo >= n) { g_err = "egg_set_actuators: body out of range"; return EGG_ERR_ARG; }
      if (re < -1 || re >= n || re == bo) { g_err = "egg_set_actuators: reaction must be -1 or another body"; return EGG_ERR_ARG; }
      if (fr != -1 && fr != bo && fr != re) { g_err = "egg_set_actuators: frame must be -1, body or reaction"; return EGG_ERR_ARG; }
      if (!std::isfinite(ax[0]) || !std::isfinite(ax[1]) || !std::isfinite(ax[2]) || (ax[0] == 0 && ax[1] == 0 && ax[2] == 0)) {
        g_err = "egg_set_actuators: an axis must be finite and not zero";
        return EGG_ERR_ARG;
      }
      cnt[bo + 1]++;
      if (re >= 0) cnt[re + 1]++;
    }
    for (int k = 0; k < n; k++) cnt[k + 1] += cnt[k];   // CSR start
    const size_t nnz = (size_t)cnt[n];
    hi.assign(3 * (size_t)m + (size_t)n + 1 + nnz, 0);
    std::copy(a->body, a->body + m, hi.begin());
    std::copy(a->reaction, a->reaction + m, hi.begin() + m);
    std::copy(a->frame, a->frame + m, hi.begin() + 2 * (size_t)m);
    std::copy(cnt.begin(), cnt.end(), hi.begin() + 3 * (size_t)m);
    int* list = hi.data() + 3 * (size_t)m + n + 1;
    for (int k = 0; k < m; k++) {   // in actuator order: every body's list is in actuator order
      list[cnt[a->body[k]]++] = k;
      if (a->reaction[k] >= 0) list[cnt[a->reaction[k]]++] = ~k;
    }
    hd.assign(a->axis, a->axis + 3 * (size_t)m);
  }
  CK(cudaSetDevice(b->device));
  // both new buffers are in place before the old ones go: a failed allocation keeps the old table
  int* qi = nullptr;
  double* qd = nullptr;
  size_t ni = 0, nd = 0;
  int r = replace_dbuf(b, qi, ni, hi.size(), hi.data());
  if (r == EGG_OK) r = replace_dbuf(b, qd, nd, hd.size(), hd.data());
  if (r != EGG_OK) {
    if (qi) dfree(b, qi, ni * sizeof(int));
    return r;
  }
  RET(replace_dbuf<int>(b, b->act_ibuf, b->act_icount, 0, nullptr));
  RET(replace_dbuf<double>(b, b->act_dbuf, b->act_dcount, 0, nullptr));
  b->act_ibuf = qi, b->act_icount = ni, b->act_dbuf = qd, b->act_dcount = nd;
  b->act = a ? EggAct{m, qi, qi + m, qi + 2 * m, qd, qi + 3 * m, qi + 3 * m + n + 1} : EggAct{};
  return EGG_OK;
}

// egg_sample_controls (std_d null: the sampler's sigma per body) and egg_sample_controls_std; ptrs
// names the entry point's device arguments.
static int sample_controls(egg_batch* b, const char* what, std::initializer_list<DevArg> ptrs, const double* mean_d, const double* std_d,
                           int horizon, unsigned long long seed, unsigned long long iteration, int first, double* u_d) {
  if (!b) return EGG_ERR_ARG;
  if (horizon < 1 || first < 0) { g_err = std::string(what) + ": horizon must be >= 1 and first >= 0"; return EGG_ERR_ARG; }
  RET(enter(b, what, INIT_LAST, ptrs, true));
  if (!b->sampler_buf) { g_err = std::string(what) + " without a sampler: call egg_set_sampler first"; return EGG_ERR_STATE; }
  CK(egg_launch_sample(b->dev, ctrl_width(b), b->sampler, mean_d, std_d, horizon, seed, iteration, first, u_d, b->stream));
  b->launches++;
  return EGG_OK;
}

int egg_sample_controls(egg_batch* b, const double* u_nom_d, int horizon, unsigned long long seed,
                        unsigned long long iteration, int first, double* u_d) {
  return sample_controls(b, "egg_sample_controls", {{u_nom_d, "u_nom_d"}, {u_d, "u_d"}}, u_nom_d, nullptr, horizon, seed, iteration,
                         first, u_d);
}

int egg_sample_controls_std(egg_batch* b, const double* mean_d, const double* std_d, int horizon, unsigned long long seed,
                            unsigned long long iteration, int first, double* u_d) {
  return sample_controls(b, "egg_sample_controls_std", {{mean_d, "mean_d"}, {std_d, "std_d"}, {u_d, "u_d"}}, mean_d, std_d, horizon,
                         seed, iteration, first, u_d);
}

// The world list of egg_gather_state and egg_gather_controls: k in [1, W] indices in [0, W).
static int check_worlds(egg_batch* b, const char* what, const int* worlds, int k) {
  const int W = b->dev.W;
  if (k < 1 || k > W) { g_err = std::string(what) + ": k must be in [1, n_worlds]"; return EGG_ERR_ARG; }
  for (int i = 0; i < k; i++)
    if (worlds[i] < 0 || worlds[i] >= W) { g_err = std::string(what) + ": world index out of range"; return EGG_ERR_ARG; }
  return EGG_OK;
}
// ... and its copy to the device, into gather_idx (allocated by the first call).
static int upload_worlds(egg_batch* b, const int* worlds, int k) {
  if (!b->gather_idx) RET(dalloc(b, &b->gather_idx, (size_t)b->dev.W));
  CK(cudaMemcpyAsync(b->gather_idx, worlds, (size_t)k * sizeof(int), cudaMemcpyHostToDevice, b->stream));
  return EGG_OK;
}

int egg_gather_controls(egg_batch* b, const double* u_d, int horizon, const int* worlds, int k, double* out_d) {
  if (!b || !worlds) return EGG_ERR_ARG;
  if (horizon < 1) { g_err = "egg_gather_controls: horizon must be >= 1"; return EGG_ERR_ARG; }
  RET(check_worlds(b, "egg_gather_controls", worlds, k));
  if ((long long)k * horizon * ctrl_width(b) > 256ll * INT_MAX) { g_err = "egg_gather_controls: too many rows"; return EGG_ERR_ARG; }
  RET(enter(b, "egg_gather_controls", INIT_LAST, {{u_d, "u_d"}, {out_d, "out_d"}}));
  RET(upload_worlds(b, worlds, k));
  CK(egg_launch_gather_controls(b->dev, ctrl_width(b), u_d, horizon, b->gather_idx, k, out_d, b->stream));
  b->launches++;
  return EGG_OK;
}

int egg_control_moments(egg_batch* b, const double* rows_d, int k, int horizon, double* out_d) {
  if (!b) return EGG_ERR_ARG;
  if (k < 1 || horizon < 1) { g_err = "egg_control_moments: k and horizon must be >= 1"; return EGG_ERR_ARG; }
  const long long L = (long long)horizon * ctrl_width(b);
  if (L > INT_MAX) { g_err = "egg_control_moments: too long a horizon"; return EGG_ERR_ARG; }
  RET(enter(b, "egg_control_moments", INIT_LAST, {{rows_d, "rows_d"}, {out_d, "out_d"}}));
  CK(egg_launch_control_moments(rows_d, k, (int)L, out_d, b->stream));
  b->launches++;
  return EGG_OK;
}

int egg_mppi_reduce(egg_batch* b, const double* u_d, int horizon, const double* cost_d, const double* baseline_d,
                    double lambda, double* out_d) {
  if (!b) return EGG_ERR_ARG;
  if (!(lambda > 0) || !std::isfinite(lambda)) { g_err = "egg_mppi_reduce: lambda must be finite and > 0"; return EGG_ERR_ARG; }
  if (horizon < 1) { g_err = "egg_mppi_reduce: horizon must be >= 1"; return EGG_ERR_ARG; }
  const int chunks = egg_mppi_chunks(b->dev.W);
  const long long cols = (long long)horizon * ctrl_width(b) + 2;
  if (chunks > 65535 || cols > INT_MAX) { g_err = "egg_mppi_reduce: too many worlds or too long a horizon"; return EGG_ERR_ARG; }
  RET(enter(b, "egg_mppi_reduce", INIT_LAST, {{u_d, "u_d"}, {cost_d, "cost_d"}, {baseline_d, "baseline_d"}, {out_d, "out_d"}}));
  const size_t need = (size_t)chunks * (size_t)cols;
  if (need > b->mppi_partial_count) RET(replace_dbuf<double>(b, b->mppi_partial, b->mppi_partial_count, need, nullptr));
  CK(egg_launch_mppi_reduce(b->dev, ctrl_width(b), u_d, horizon, cost_d, baseline_d, lambda, b->mppi_partial, out_d, b->stream));
  b->launches += 2;
  return EGG_OK;
}

int egg_gather_state(egg_batch* b, const int* worlds, int k, double* out_d) {
  if (!b || !worlds || !out_d) return EGG_ERR_ARG;
  RET(check_worlds(b, "egg_gather_state", worlds, k));
  RET(enter(b, "egg_gather_state", INIT_FIRST, {{out_d, "out_d"}}));
  RET(upload_worlds(b, worlds, k));
  CK(egg_launch_gather_state(b->dev, b->gather_idx, k, out_d, b->stream));
  b->launches++;
  return EGG_OK;
}

int egg_seed_state(egg_batch* b, const double* in_d, int k, int first) {
  if (!b || !in_d) return EGG_ERR_ARG;
  if (k < 1 || k > b->dev.W || first < 0) { g_err = "egg_seed_state: k must be in [1, n_worlds] and first >= 0"; return EGG_ERR_ARG; }
  RET(enter(b, "egg_seed_state", INIT_FIRST, {{in_d, "in_d"}}));
  CK(egg_launch_seed_state(b->dev, in_d, k, first, b->stream));
  b->launches++;
  return EGG_OK;
}

int egg_update_contacts(egg_batch* b) {
  if (!b) return EGG_ERR_ARG;
  if (!b->initialised) { g_err = "egg_update_contacts before egg_init"; return EGG_ERR_STATE; }
  CK(cudaSetDevice(b->device));
  CK(egg_launch_collide(b->dev, b->stream));
  b->launches++;
  return EGG_OK;
}

int egg_get_static(egg_batch* b, double* minv_lin, double* minv_ang, double* f_ext) {
  if (!b) return EGG_ERR_ARG;
  CK(cudaSetDevice(b->device));
  const int n = b->dev.n;
  if (minv_lin) RET(download(b, minv_lin, n, 1, b->dev.stat, EGG_STAT, 0));
  if (minv_ang) RET(download(b, minv_ang, n, 9, b->dev.stat, EGG_STAT, 1));
  if (f_ext) RET(download(b, f_ext, n, 6, b->dev.stat, EGG_STAT, 10));
  return EGG_OK;
}

int egg_snapshot(egg_batch* b) {
  if (!b) return EGG_ERR_ARG;
  CK(cudaSetDevice(b->device));
  const size_t cnt = (size_t)b->dev.W * EGG_DYN * b->dev.n;
  if (!b->snap) {
    int r = dalloc(b, &b->snap, cnt);
    if (r != EGG_OK) return r;
  }
  CK(cudaMemcpyAsync(b->snap, b->dev.dyn, cnt * sizeof(double), cudaMemcpyDeviceToDevice, b->stream));
  return EGG_OK;
}
int egg_restore(egg_batch* b) {
  if (!b) return EGG_ERR_ARG;
  if (!b->snap) { g_err = "egg_restore before egg_snapshot"; return EGG_ERR_STATE; }
  CK(cudaSetDevice(b->device));
  const size_t cnt = (size_t)b->dev.W * EGG_DYN * b->dev.n;
  CK(cudaMemcpyAsync(b->dev.dyn, b->snap, cnt * sizeof(double), cudaMemcpyDeviceToDevice, b->stream));
  return EGG_OK;
}

int egg_get_bodies(egg_batch* b, double* p, double* R, double* v, double* w) {
  if (!b) return EGG_ERR_ARG;
  CK(cudaSetDevice(b->device));
  const int n = b->dev.n;
  if (p) RET(download(b, p, n, 3, b->dev.dyn, EGG_DYN, 0));
  if (R) RET(download(b, R, n, 9, b->dev.dyn, EGG_DYN, 3));
  if (v) RET(download(b, v, n, 3, b->dev.dyn, EGG_DYN, 12));
  if (w) RET(download(b, w, n, 3, b->dev.dyn, EGG_DYN, 15));
  CK(cudaStreamSynchronize(b->stream));
  return EGG_OK;
}

// Contact taps of worlds [first, first + count): the geometry is transposed from the device's
// [world][7][max_contacts] layout to the host's [world][max_contacts][3] by the unpack kernel, in
// chunks of as many worlds as fit the staging buffer (no host-side pass over the data).
int egg_get_contacts_range(egg_batch* b, int first, int nworlds, int* count, int* i0, int* i1, double* pos, double* nrm,
                           double* depth, int* code, double* lambda, int* row_state) {
  if (!b || first < 0 || nworlds < 0 || first + nworlds > b->dev.W) return EGG_ERR_ARG;
  CK(cudaSetDevice(b->device));
  const EggDev& d = b->dev;
  const size_t W = (size_t)nworlds, mc = d.maxc, f = (size_t)first;
  if (W == 0) return EGG_OK;
  if (count) CK(cudaMemcpyAsync(count, d.c_count + f, W * sizeof(int), cudaMemcpyDeviceToHost, b->stream));
  if (i0) CK(cudaMemcpyAsync(i0, d.c_i0 + f * mc, W * mc * sizeof(int), cudaMemcpyDeviceToHost, b->stream));
  if (i1) CK(cudaMemcpyAsync(i1, d.c_i1 + f * mc, W * mc * sizeof(int), cudaMemcpyDeviceToHost, b->stream));
  if (code) CK(cudaMemcpyAsync(code, d.c_code + f * mc, W * mc * sizeof(int), cudaMemcpyDeviceToHost, b->stream));
  if (lambda) CK(cudaMemcpyAsync(lambda, d.lam_out + f * 3 * d.nrec, W * 3 * d.nrec * sizeof(double), cudaMemcpyDeviceToHost, b->stream));
  if (row_state) CK(cudaMemcpyAsync(row_state, d.row_state + f * 3 * d.nrec, W * 3 * d.nrec * sizeof(int), cudaMemcpyDeviceToHost, b->stream));
  if (pos || nrm || depth) {
    size_t chunk = b->stage_bytes / (mc * 3 * sizeof(double));
    if (chunk == 0) { g_err = "staging buffer smaller than one world's contact geometry"; return EGG_ERR_UNSUPPORTED; }
    struct { double* host; int comps, off; } part[3] = {{pos, 3, 0}, {nrm, 3, 3}, {depth, 1, 6}};
    for (size_t w0 = 0; w0 < W; w0 += chunk) {
      const size_t nw = (W - w0 < chunk) ? W - w0 : chunk;
      for (auto& pt : part) {
        if (!pt.host) continue;
        CK(egg_launch_unpack((int)nw, b->stage, (int)mc, pt.comps, d.c_geom + (f + w0) * 7 * mc, 7, pt.off, b->stream));
        b->launches++;
        CK(cudaMemcpyAsync(pt.host + w0 * mc * pt.comps, b->stage, nw * mc * pt.comps * sizeof(double), cudaMemcpyDeviceToHost, b->stream));
        CK(cudaStreamSynchronize(b->stream));      // the staging buffer is reused by the next part
      }
    }
  }
  CK(cudaStreamSynchronize(b->stream));
  return EGG_OK;
}

int egg_get_contacts(egg_batch* b, int* count, int* i0, int* i1, double* pos, double* nrm,
                     double* depth, int* code, double* lambda, int* row_state) {
  if (!b) return EGG_ERR_ARG;
  return egg_get_contacts_range(b, 0, b->dev.W, count, i0, i1, pos, nrm, depth, code, lambda, row_state);
}

int egg_get_pair_hits_range(egg_batch* b, int first, int nworlds, int* n_hits, int* pi, int* pj, int* code, int* count, int max_pairs) {
  if (!b || !n_hits || first < 0 || nworlds < 0 || first + nworlds > b->dev.W) return EGG_ERR_ARG;
  const EggDev& d = b->dev;
  if (!d.pair_code) { g_err = "egg_get_pair_hits needs desc.taps = 1"; return EGG_ERR_STATE; }
  CK(cudaSetDevice(b->device));
  const size_t W = (size_t)nworlds, P = d.P, f = (size_t)first;
  if (W == 0 || P == 0) { for (size_t w = 0; w < W; w++) n_hits[w] = 0; return EGG_OK; }
  std::vector<unsigned char> pc(W * P), pn(W * P);
  CK(cudaMemcpyAsync(pc.data(), d.pair_code + f * P, W * P, cudaMemcpyDeviceToHost, b->stream));
  CK(cudaMemcpyAsync(pn.data(), d.pair_cnt + f * P, W * P, cudaMemcpyDeviceToHost, b->stream));
  CK(cudaStreamSynchronize(b->stream));
  for (size_t w = 0; w < W; w++) {
    int h = 0;
    size_t q = 0;
    for (int i = 0; i < d.n; i++)
      for (int j = i + 1; j < d.n; j++, q++) {
        if (!pc[w * P + q]) continue;
        if (h < max_pairs) {
          if (pi) pi[w * max_pairs + h] = i;
          if (pj) pj[w * max_pairs + h] = j;
          if (code) code[w * max_pairs + h] = pc[w * P + q];
          if (count) count[w * max_pairs + h] = pn[w * P + q];
        }
        h++;
      }
    n_hits[w] = h;
  }
  return EGG_OK;
}

int egg_get_pair_hits(egg_batch* b, int* n_hits, int* pi, int* pj, int* code, int* count, int max_pairs) {
  if (!b) return EGG_ERR_ARG;
  return egg_get_pair_hits_range(b, 0, b->dev.W, n_hits, pi, pj, code, count, max_pairs);
}

int egg_get_status(egg_batch* b, int* status, int* stats, double* residual) {
  if (!b) return EGG_ERR_ARG;
  CK(cudaSetDevice(b->device));
  const size_t W = b->dev.W;
  if (status) CK(cudaMemcpyAsync(status, b->dev.status, W * sizeof(int), cudaMemcpyDeviceToHost, b->stream));
  if (stats) CK(cudaMemcpyAsync(stats, b->dev.stats, W * 8 * sizeof(int), cudaMemcpyDeviceToHost, b->stream));
  if (residual) CK(cudaMemcpyAsync(residual, b->dev.resid, W * sizeof(double), cudaMemcpyDeviceToHost, b->stream));
  CK(cudaStreamSynchronize(b->stream));
  return EGG_OK;
}

int egg_get_debug_counters(egg_batch* b, unsigned long long* out32, int reset) {
  if (!b || !out32) return EGG_ERR_ARG;
  CK(cudaSetDevice(b->device));
  CK(cudaMemcpyAsync(out32, b->dev.dbg, 32 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, b->stream));
  if (reset) CK(cudaMemsetAsync(b->dev.dbg, 0, 32 * sizeof(unsigned long long), b->stream));
  CK(cudaStreamSynchronize(b->stream));
  return EGG_OK;
}

int egg_get_dense_work(egg_batch* b, double* flops) {
  if (!b || !flops) return EGG_ERR_ARG;
  if (!b->dev.work) { g_err = "egg_get_dense_work: the batch was not created with the dense solver"; return EGG_ERR_STATE; }
  CK(cudaSetDevice(b->device));
  CK(cudaMemcpyAsync(flops, b->dev.work, (size_t)b->dev.W * sizeof(double), cudaMemcpyDeviceToHost, b->stream));
  CK(cudaStreamSynchronize(b->stream));
  return EGG_OK;
}

int egg_rollout_costs(egg_batch* b, double* cost_d) {
  RET(enter(b, "egg_rollout_costs", INIT_NONE, {{cost_d, "cost_d"}}));
  CK(egg_launch_costs(b->dev, cost_d, b->stream));
  b->launches++;
  return EGG_OK;
}

}  // extern "C"
