// Internal device-side layout of an egg_batch and small FP64 vector helpers.
//
// HBM layout (FP64, indices int32), W worlds of n bodies, nj joints, capacity maxc contacts:
//   dyn    [W][18][n]   p(3) R(9, row-major) v(3) w(3)          Body state, body.h:79-84
//   stat   [W][16][n]   1/m, (R I_b R^T)^-1 (9), f_ext (6)      ensembles.cc:202-222 (frozen at init)
//   bpar   [W][14][n]   side(3) m I_b(9) shape                  body.h:81,85,91 (shape: 0 box, 1 sphere, 2 capsule; side = dims)
//   joints [W][nj] i0,i1 ; jc [W][6][nj] c0(3) c1(3)            joints.h:26-28
//   contacts: c_i0,c_i1,c_code [W][maxc]; c_geom [W][7][maxc] pos(3) nrm(3) depth
//   records [W][nrec] x 240 B in dependency-level order; inside one level chunk (<= 32 blocks,
//           one solver stage) the 15 16-byte pieces are stored piece-major: [piece][block], so a
//           stage is one contiguous TMA bulk copy and lanes read consecutive 16-byte words;
//           lam [W][nrec][3]
// The body index is the fastest-varying one inside a world so that a warp working on one world
// reads/writes contiguous 8-byte lanes; a world is one contiguous chunk (TMA-bulk friendly).
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <cmath>

#define EGG_DYN 18
#define EGG_STAT 16
#define EGG_BPAR 14
#define EGG_REC 30          // doubles per constraint record (15 x 16-byte pieces = 240 B)
#define EGG_PIECES 15
#define EGG_MAX_POLY 12
#define EGG_MAX_PAIR_CONTACTS 10

// Record field offsets (doubles).
#define REC_RC 0            // 9: contact frame (rows = tangent0, tangent1, normal); joints: -I
#define REC_R0 9            // 3: pos - p(i0)   (joints: R0 c0)
#define REC_R1 12           // 3: pos - p(i1)   (joints: R1 c1)
#define REC_DOFF 15         // 3: d10 d20 d21 of the 3x3 diagonal block of J M^-1 J^T
#define REC_DDIAG 18        // 3: d00 d11 d22 (no cfm)
#define REC_INVA 21         // 3: 1 / (dkk + cfm)
#define REC_RHS 24          // 3
#define REC_IDX 27          // int2: i0, i1
#define REC_META 28         // int2: original constraint index, clamp kind

// Clamp kinds of a 3-row block.
#define KIND_EQUALITY 0     // joints: no projection
#define KIND_CONTACT 1      // rows 0,1 in [-1,1], row 2 in [0,inf)  (contact.cc:103-113)

struct EggParams {
  double erp, cfm, tol, min_dist;
  double g[3];
  int k_max, solver, quirks, cfm_mode;
};

// Development overrides of the kernel selection, read from the environment by egg_create and kept
// with the batch, so that batches of one process can run different instances.  Unset variables
// take the defaults below; lpw, run_cap, collide_nt and records_nt = 0 leave the choice to the
// selection rules of the launchers.
struct EggSel {
  int lpw;           // EGG_PGS_LPW: lanes per world 1 / 2 / 4 / 8 / 16 of the group stream
  int min_warps;     // EGG_PGS_MIN_WARPS_PER_SM: warps per SM the LPW rule aims for (default 3)
  int runs;          // EGG_PGS_RUNS: -1 unset, 0 off, 1 on (overrides EGG_OPT_PGS_RUNS)
  int run_cap;       // EGG_PGS_RUN_CAP: runs per world and stage of the run format
  int target_ctas;   // EGG_PGS_TARGET_CTAS: resident CTAs per SM the run cap is sized for (default 11)
  int collide_nt;    // EGG_COLLIDE_NT: narrowphase threads per world
  int records_nt;    // EGG_RECORDS_NT: record-assembly threads per world of the group stream / run format
  int ctas_per_sm;   // EGG_PGS_CTAS_PER_SM: cap on resident solve CTAs per SM (grid size only)
  int pf;            // EGG_PGS_PF: L2 prefetch depth of the solve in 4 KB rounds (default 3)
};

struct EggDev {
  int W, n, nj, maxc, P, nrec;   // P = n(n-1)/2, nrec = nj + maxc
  double* dyn;
  double* stat;
  double* bpar;
  double* minv_aos;           // [W][n+1][10] = 1/m, I^-1 per body (row n = 0: the dummy 'world' body)
  int* j_i0;
  int* j_i1;
  double* jc;
  int* c_count;
  int* c_i0;
  int* c_i1;
  int* c_code;
  double* c_geom;
  unsigned char* pair_code;   // taps, may be null: [W][P]
  unsigned char* pair_cnt;
  double* rec;
  double* lam;                // [W][nrec][3] slot order during the solve (Jacobi / SOR only, else null)
  double* lam2;               // second multiplier buffer (Jacobi / SOR only, else null)
  double* lam_out;            // [W][3*nrec] row order (joints then contacts)
  int* row_state;             // [W][3*nrec]
  int* slot_of;               // [W][nrec] record slot of reference constraint c (Jacobi / SOR only, else null)
  int* level_start;           // [W][nrec+1] start slot of every stage of the per-world record order (null with the group stream)
  int* n_levels;              // [W] number of stages
  int* status;                // [W]
  int* stats;                 // [W][8]
  double* resid;              // [W]
  double* work;               // [W] algorithmic FP64 operations of the last dense solve (dense solver only, else null)
  double* cost0;              // [W][2]
  double* minv_iso;           // [W][n+1][2] = 1/m, 1/c per body when every inverse inertia is c^-1 I3 (row n = 0)
  int* iso_flag;              // [1] device: 1 while every body seen by egg_init was isotropic
  int iso;                    // host copy of iso_flag, valid after the first step following egg_init
  // group-stream assembly of the default PGS variant (egg_pgs_stream.cu)
  int blkb;                   // stream bytes per block: 32 (multipliers) + 176 (FP64 record) or 112 (precision = 32 record)
  int lpw;                    // lanes per world = stage cap; G = 32 / lpw worlds share a warp and a record stream
  int rmax;                   // 0: one block per lane and stage (egg_pgs_stream.cu); >= 1: run format, a lane carries a run of up to rmax
                              //    consecutive blocks on the same body pair through a stage (egg_pgs_runs.cu)
  unsigned* st_runs;          // [W][nrec] run lengths of a world's stage, 4 bits per lane of the world (run format only, else null)
  int run_cap;                // runs per world and stage of the run format (<= lpw; bounded by the staging buffer)
  int* c_pos;                 // [W][nrec] stage << 8 | index inside the stage, per constraint
  unsigned char* st_cnt;      // [W][nrec] blocks per stage
  unsigned* round_off;        // [groups][nrec+1] byte offset of every round inside the group stream
  int* grp_info;              // [groups][4] rounds, blocks in round 0, stream bytes
  int* work_ctr;              // [4] world-group queue of the persistent solve kernel
  unsigned long long* dbg;    // [32] debug / phase-timing counters (written only by builds with EGG_DENSE_TIMING)
  int rec_fmt;                // 0: D diagonal in REC_DDIAG, multipliers in lam[]; 1: multipliers in REC_DDIAG, next-stage count in slot 29 (stream variant)
  EggParams prm;
  EggSel sel;
};

struct d3 {
  double x, y, z;
};
__host__ __device__ inline d3 mk3(double x, double y, double z) { d3 r; r.x = x; r.y = y; r.z = z; return r; }
__host__ __device__ inline d3 operator+(d3 a, d3 b) { return mk3(a.x + b.x, a.y + b.y, a.z + b.z); }
__host__ __device__ inline d3 operator-(d3 a, d3 b) { return mk3(a.x - b.x, a.y - b.y, a.z - b.z); }
__host__ __device__ inline d3 operator-(d3 a) { return mk3(-a.x, -a.y, -a.z); }
__host__ __device__ inline d3 operator*(d3 a, double s) { return mk3(a.x * s, a.y * s, a.z * s); }
__host__ __device__ inline d3 operator*(double s, d3 a) { return mk3(a.x * s, a.y * s, a.z * s); }
__host__ __device__ inline d3 operator/(d3 a, double s) { return mk3(a.x / s, a.y / s, a.z / s); }
__host__ __device__ inline double dot3(d3 a, d3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
__host__ __device__ inline d3 cross3(d3 a, d3 b) {
  return mk3(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x);
}
__host__ __device__ inline double norm3(d3 a) { return sqrt(dot3(a, a)); }
__host__ __device__ inline double get3(d3 a, int i) { return i == 0 ? a.x : (i == 1 ? a.y : a.z); }
__host__ __device__ inline void set3(d3& a, int i, double v) {
  if (i == 0) a.x = v; else if (i == 1) a.y = v; else a.z = v;
}
// Row-major 3x3 in a flat array m[9].
__host__ __device__ inline d3 mcol(const double* m, int c) { return mk3(m[c], m[3 + c], m[6 + c]); }
__host__ __device__ inline d3 mrow(const double* m, int r) { return mk3(m[3 * r], m[3 * r + 1], m[3 * r + 2]); }
__host__ __device__ inline d3 mmulv(const double* m, d3 v) {
  return mk3(m[0] * v.x + m[1] * v.y + m[2] * v.z, m[3] * v.x + m[4] * v.y + m[5] * v.z,
             m[6] * v.x + m[7] * v.y + m[8] * v.z);
}
__host__ __device__ inline d3 mtmulv(const double* m, d3 v) {
  return mk3(m[0] * v.x + m[3] * v.y + m[6] * v.z, m[1] * v.x + m[4] * v.y + m[7] * v.z,
             m[2] * v.x + m[5] * v.y + m[8] * v.z);
}
__host__ __device__ inline void mmulm(const double* a, const double* b, double* o) {
  for (int i = 0; i < 3; i++)
    for (int j = 0; j < 3; j++) o[3 * i + j] = a[3 * i] * b[j] + a[3 * i + 1] * b[3 + j] + a[3 * i + 2] * b[6 + j];
}
__host__ __device__ inline double sign1(double a) { return (a >= 0) ? 1.0 : -1.0; }

// Launch wrappers (defined in the .cu files).  Every wrapper returns the first CUDA error of its
// attribute / occupancy / memset / launch calls (cudaSuccess otherwise); egg_capi.cu turns it into
// EGG_ERR_CUDA with the wrapper's name in egg_last_error().
cudaError_t egg_launch_collide(const EggDev& d, cudaStream_t s);
cudaError_t egg_launch_init(const EggDev& d, cudaStream_t s);
cudaError_t egg_launch_clear_contacts(const EggDev& d, cudaStream_t s);
cudaError_t egg_launch_assemble(const EggDev& d, double dt, cudaStream_t s);
// mu: the [W] Coulomb friction coefficients of egg_set_friction (device), null = BOX friction.  A
// kernel argument of its own rather than a member of EggDev: the parameter layout of the kernels
// that do not read it stays put.
cudaError_t egg_launch_solve_pgs(const EggDev& d, double dt, const double* mu, cudaStream_t s);
cudaError_t egg_launch_solve_pgs_stream(const EggDev& d, double dt, const double* mu, cudaStream_t s);
cudaError_t egg_launch_solve_pgs_runs(const EggDev& d, double dt, cudaStream_t s);
int egg_run_cap(const EggDev& d);
int egg_runs_rmax(const EggDev& d);
size_t egg_runs_smem(const EggDev& d);
cudaError_t egg_launch_assemble_runs_tail(const EggDev& d, double dt, cudaStream_t s);
cudaError_t egg_launch_assemble_stream(const EggDev& d, double dt, cudaStream_t s);
size_t egg_stream_rec_bytes(int W, int nrec, int lpw);
int egg_stream_blkb(int precision);
int egg_stage_cap(const EggDev& d);
// Threads per world of the instance each pre-solve launcher runs for this batch (egg_get_kernel_config).
int egg_collide_threads(const EggDev& d);
int egg_records_threads(const EggDev& d);
int egg_assemble_threads(const EggDev& d);
cudaError_t egg_launch_solve_iter(const EggDev& d, double dt, int solver, cudaStream_t s);
cudaError_t egg_launch_costs(const EggDev& d, double* cost_d, cudaStream_t s);
cudaError_t egg_launch_pack(int W, const double* aos, int per_world, int comps, double* soa, int soa_comps, int comp_off, cudaStream_t s);
cudaError_t egg_launch_unpack(int W, double* aos, int per_world, int comps, const double* soa, int soa_comps, int comp_off, cudaStream_t s);
// one control slice u [W][n][6] (device) -> the f_ext slot of stat
cudaError_t egg_launch_fext_slice(const EggDev& d, const double* u, cudaStream_t s);
// dyn of worlds[0..k) (device int array) -> out [k][n][18]; dyn of world w <- in [(first + w) mod k][n][18]
cudaError_t egg_launch_gather_state(const EggDev& d, const int* worlds, int k, double* out, cudaStream_t s);
cudaError_t egg_launch_seed_state(const EggDev& d, const double* in, int k, int first, cudaStream_t s);
// Device copy of egg_set_cost, shared by all worlds and stored component-major ([c][n], the body
// index fastest, like dyn) so that the lanes of a warp read consecutive words.
struct EggCost {
  const double* q_run;    // [18][n]
  const double* l_run;    // [18][n]
  const double* u_run;    // [6][n], or [m] with an actuator table
  const double* q_term;   // [18][n]
  const double* l_term;   // [18][n]
  const double* x_ref;    // [ref_steps][18][n]
  int ref_steps;
};
// egg_launch_fext_slice that also adds the running cost at (x_t, u_t) to cost[W] (stores it at t = 0);
// the terminal term at x_horizon is added after the last step
cudaError_t egg_launch_fext_slice_cost(const EggDev& d, const double* u, const EggCost& c, int t, double* cost, cudaStream_t s);
cudaError_t egg_launch_cost_terminal(const EggDev& d, const EggCost& c, int horizon, double* cost, cudaStream_t s);
// Device copy of egg_set_actuators, shared by all worlds.  start / list: per body b, the actuators
// that touch it in actuator order, list[start[b] .. start[b + 1]), a for +tau (b = body[a]) and ~a
// for -tau (b = reaction[a]).
struct EggAct {
  int m;
  const int* body;        // [m]
  const int* reaction;    // [m], -1 = none
  const int* frame;       // [m], -1 = world
  const double* axis;     // [m][3]
  const int* start;       // [n + 1]
  const int* list;        // [start[n]]
};
// Actuator mode: one control row u [W][m] (device) -> the f_ext slot of stat, m g plus the actuator
// torques; with c (not null) the running cost of step t as egg_launch_fext_slice_cost adds it, the
// control term sum_a u_run[a] u_a^2 (c->u_run is [m]).
cudaError_t egg_launch_actuate(const EggDev& d, const EggAct& a, const double* u, const EggCost* c, int t, double* cost, cudaStream_t s);
// Device copy of egg_set_sampler: sigma, u_lo, u_hi, each one control row [c] (+-inf for no bound);
// c = 6 n ([n][6]) with body wrenches, m with an actuator table.
struct EggSampler {
  const double* sigma;
  const double* lo;
  const double* hi;
};
// Sampling (egg_sample_controls, egg_sample_controls_std): u [H][W][c] <- clamp(mean [H][c] + sigma eps)
// with sm.sigma per element of the row, or with the per-step std_dev [H][c] in its place when std_dev
// is not null.  c is the control row width.
cudaError_t egg_launch_sample(const EggDev& d, int c, const EggSampler& sm, const double* mean, const double* std_dev, int horizon,
                              unsigned long long seed, unsigned long long iteration, int first, double* u, cudaStream_t s);
// MPPI (egg_mppi_reduce): out [H c + 2] <- sum_w omega_w u[t][w], sum omega, sum omega^2 through
// partial [chunks][H c + 2]
int egg_mppi_chunks(int W);   // stage-1 chunks of egg_launch_mppi_reduce: partial holds chunks x (H c + 2) doubles
cudaError_t egg_launch_mppi_reduce(const EggDev& d, int c, const double* u, int horizon, const double* cost, const double* baseline,
                                   double lambda, double* partial, double* out, cudaStream_t s);
// CEM (egg_gather_controls, egg_control_moments): out [k][H][c] <- u[t][worlds[i]];
// out [2][L] <- mean and population std of the columns of rows [k][L]
cudaError_t egg_launch_gather_controls(const EggDev& d, int c, const double* u, int horizon, const int* worlds, int k, double* out,
                                       cudaStream_t s);
cudaError_t egg_launch_control_moments(const double* rows, int k, int L, double* out, cudaStream_t s);
// Dynamic shared memory each kernel family needs for this batch shape (checked against the device
// limit in egg_create, so that an unsupported shape fails there with a clear message).
size_t egg_collide_smem(const EggDev& d);
size_t egg_assemble_smem(const EggDev& d);
size_t egg_stream_smem(const EggDev& d);
size_t egg_iter_smem(const EggDev& d);
// FIRST(e, call): keep the first error of a sequence of CUDA calls.
#define EGG_FIRST(e, call) do { cudaError_t e2__ = (call); if ((e) == cudaSuccess) (e) = e2__; } while (0)
