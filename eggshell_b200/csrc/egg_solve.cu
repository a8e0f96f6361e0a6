// Init, rollout costs, MPC control slices and state exchange, AoS<->SoA staging and the FP64
// roofline probe (assembly + PGS: egg_pgs.cu).
//
// Replaces (per world):
//   egg_init_kernel        Ensemble::Init pieces          ensembles.cc:24-29, 202-232
//   egg_init_check_kernel  CheckInitialConditions         ensembles.cc:224-232
#include "egg_internal.cuh"

namespace {

__device__ inline void inverse3(const double* m, double* r) {
  double c00 = m[4] * m[8] - m[5] * m[7];
  double c01 = m[5] * m[6] - m[3] * m[8];
  double c02 = m[3] * m[7] - m[4] * m[6];
  double det = m[0] * c00 + m[1] * c01 + m[2] * c02;
  double id = 1.0 / det;
  r[0] = c00 * id; r[3] = c01 * id; r[6] = c02 * id;
  r[1] = (m[2] * m[7] - m[1] * m[8]) * id;
  r[4] = (m[0] * m[8] - m[2] * m[6]) * id;
  r[7] = (m[1] * m[6] - m[0] * m[7]) * id;
  r[2] = (m[1] * m[5] - m[2] * m[4]) * id;
  r[5] = (m[2] * m[3] - m[0] * m[5]) * id;
  r[8] = (m[0] * m[4] - m[1] * m[3]) * id;
}

// ---------------------------------------------------------------------------------------------
// Init: thread per (world, body).
__global__ void egg_init_kernel(EggDev d) {
  const int n = d.n;
  const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (gid >= (long long)d.W * n) return;
  const int w = (int)(gid / n), b = (int)(gid % n);
  const double* dyn = d.dyn + (size_t)w * EGG_DYN * n;
  const double* bp = d.bpar + (size_t)w * EGG_BPAR * n;
  double* st = d.stat + (size_t)w * EGG_STAT * n;
  double R[9], I[9], RI[9], Ig[9], Rt[9], inv[9];
  for (int k = 0; k < 9; k++) { R[k] = dyn[(3 + k) * n + b]; I[k] = bp[(4 + k) * n + b]; }
  for (int i = 0; i < 3; i++) for (int j = 0; j < 3; j++) Rt[3 * i + j] = R[3 * j + i];
  mmulm(R, I, RI);
  mmulm(RI, Rt, Ig);           // I_g = (R I) R^T, body.h:58
  inverse3(Ig, inv);           // ensembles.cc:210
  // Isotropic bodies (I_b = c I3 exactly: every body of the reference's Chain / Cairn scenes):
  // R (c I3) R^T is c I3 up to rounding, and so is its inverse.  When the computed inverse agrees
  // with (1/c) I3 to 1e-13 relative it is replaced by exactly that, so that the solver can keep
  // two doubles per body; a body that is not isotropic clears the batch-wide flag (bit 0) and the
  // general kernels run.  EGG_OPT_EXACT_INERTIA (quirks bit 4) keeps the matrix as computed.
  {
    const bool diag = I[1] == 0.0 && I[2] == 0.0 && I[3] == 0.0 && I[5] == 0.0 && I[6] == 0.0 && I[7] == 0.0 && I[0] == I[4] && I[0] == I[8];
    const double ic = 1.0 / I[0];
    double dev = fmax(fmax(fabs(inv[0] - ic), fabs(inv[4] - ic)), fabs(inv[8] - ic));
    dev = fmax(dev, fmax(fmax(fabs(inv[1]), fabs(inv[2])), fmax(fabs(inv[3]), fabs(inv[5]))));
    dev = fmax(dev, fmax(fabs(inv[6]), fabs(inv[7])));
    const bool iso = !(d.prm.quirks & 4) && diag && dev <= 1e-13 * fabs(ic);
    if (iso) {
      for (int k = 0; k < 9; k++) inv[k] = 0.0;
      inv[0] = inv[4] = inv[8] = ic;
    } else {
      atomicAnd(d.iso_flag, 0);
    }
    d.minv_iso[((size_t)w * (n + 1) + b) * 2 + 1] = ic;
  }
  const double m = bp[3 * n + b];
  st[0 * n + b] = 1.0 / m;     // ensembles.cc:207
  for (int k = 0; k < 9; k++) st[(1 + k) * n + b] = inv[k];
  {
    double* ma = d.minv_aos + ((size_t)w * (n + 1) + b) * 10;
    ma[0] = 1.0 / m;
    for (int k = 0; k < 9; k++) ma[1 + k] = inv[k];
    d.minv_iso[((size_t)w * (n + 1) + b) * 2] = 1.0 / m;
  }
  d3 wv = mk3(dyn[15 * n + b], dyn[16 * n + b], dyn[17 * n + b]);
  // f_ext = [m g ; ((-[w]x) I_g) w]   ensembles.cc:218-220
  double ncm[9] = {-0.0, wv.z, -wv.y, -wv.z, -0.0, wv.x, wv.y, -wv.x, -0.0};
  double t[9];
  mmulm(ncm, Ig, t);
  d3 tq = mmulv(t, wv);
  st[10 * n + b] = m * d.prm.g[0];
  st[11 * n + b] = m * d.prm.g[1];
  st[12 * n + b] = m * d.prm.g[2];
  st[13 * n + b] = tq.x; st[14 * n + b] = tq.y; st[15 * n + b] = tq.z;
  if (b == 0) {
    d.cost0[2 * w] = dyn[0 * n];       // x of body 0
    d.cost0[2 * w + 1] = dyn[2 * n];   // z of body 0
    d.status[w] = 0;
    for (int k = 0; k < 8; k++) d.stats[(size_t)w * 8 + k] = 0;
    d.resid[w] = 0;
    d.c_count[w] = 0;
  }
}

// Bit 1 of the isotropy flag: every body of the batch has the same (1/m, 1/c) as body 0 of world 0.
__global__ void egg_iso_uniform_kernel(EggDev d) {
  const int n = d.n;
  const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (gid >= (long long)d.W * n) return;
  const int w = (int)(gid / n), b = (int)(gid % n);
  const double* mi = d.minv_iso + ((size_t)w * (n + 1) + b) * 2;
  if (mi[0] != d.minv_iso[0] || mi[1] != d.minv_iso[1]) atomicAnd(d.iso_flag, ~2);
}

// CheckInitialConditions (ensembles.cc:224-232): every joint error component within 1e-9.
__global__ void egg_init_check_kernel(EggDev d) {
  const int n = d.n, nj = d.nj;
  const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (gid >= (long long)d.W * nj) return;
  const int w = (int)(gid / nj), k = (int)(gid % nj);
  const double* dyn = d.dyn + (size_t)w * EGG_DYN * n;
  const double* jc = d.jc + (size_t)w * 6 * nj;
  const int i0 = d.j_i0[(size_t)w * nj + k], i1 = d.j_i1[(size_t)w * nj + k];
  double R0[9];
  for (int c = 0; c < 9; c++) R0[c] = dyn[(3 + c) * n + i0];
  d3 e = mk3(dyn[i0], dyn[n + i0], dyn[2 * n + i0]) + mmulv(R0, mk3(jc[k], jc[nj + k], jc[2 * nj + k]));
  d3 c1 = mk3(jc[3 * nj + k], jc[4 * nj + k], jc[5 * nj + k]);
  if (i1 < 0) e = e - c1;
  else {
    double R1[9];
    for (int c = 0; c < 9; c++) R1[c] = dyn[(3 + c) * n + i1];
    e = e - mk3(dyn[i1], dyn[n + i1], dyn[2 * n + i1]) - mmulv(R1, c1);
  }
  if (fabs(e.x) > 1e-9 || fabs(e.y) > 1e-9 || fabs(e.z) > 1e-9) atomicOr(&d.status[w], 4 /*EGG_ST_BAD_INIT*/);
}

// After the init-time narrowphase pass (run only for its joint-joint conflict scan): the reference's
// contact list is empty until the first Step / UpdateContacts (Ensemble::Init never calls
// UpdateContacts, ensembles.cc:24-29), so the list, its statistics and a contact-overflow flag of
// that pass are dropped again.
__global__ void egg_clear_contacts_kernel(EggDev d) {
  const int w = blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= d.W) return;
  d.c_count[w] = 0;
  int* st = d.stats + (size_t)w * 8;
  st[0] = 0; st[1] = 0; st[2] = 3 * d.nj; st[3] = 0;
  d.status[w] &= ~8;
}

__global__ void egg_cost_kernel(EggDev d, double* cost) {
  const int w = blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= d.W) return;
  const double* dyn = d.dyn + (size_t)w * EGG_DYN * d.n;
  double dx = dyn[0] - d.cost0[2 * w];
  double dz = dyn[2 * d.n] - d.cost0[2 * w + 1];
  cost[w] = -dx + 10.0 * dz * dz;
}

// AoS [W][per_world][comps] (host order) -> SoA [W][comps_total][per_world] at component offset.
__global__ void egg_pack_kernel(const double* aos, int W, int per_world, int comps, double* soa, int soa_comps, int comp_off) {
  const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long total = (long long)W * per_world * comps;
  if (gid >= total) return;
  const int c = (int)(gid % comps);
  const long long t = gid / comps;
  const int b = (int)(t % per_world);
  const int w = (int)(t / per_world);
  soa[((size_t)w * soa_comps + comp_off + c) * per_world + b] = aos[gid];
}
__global__ void egg_unpack_kernel(double* aos, int W, int per_world, int comps, const double* soa, int soa_comps, int comp_off) {
  const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long total = (long long)W * per_world * comps;
  if (gid >= total) return;
  const int c = (int)(gid % comps);
  const long long t = gid / comps;
  const int b = (int)(t % per_world);
  const int w = (int)(t / per_world);
  aos[gid] = soa[((size_t)w * soa_comps + comp_off + c) * per_world + b];
}

// One slice of a control schedule, AoS u [W][n][6] -> the f_ext components 10..15 of stat [W][16][n].
// One thread per (w, component, body) with the body fastest: the writes are coalesced, and the reads
// of a warp (48-byte stride) share their sectors with the warps of the neighbouring components.
__global__ void egg_fext_slice_kernel(const double* u, int W, int n, double* stat) {
  const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (gid >= (long long)W * 6 * n) return;
  const int b = (int)(gid % n);
  const long long t = gid / n;
  const int c = (int)(t % 6);
  const long long w = t / 6;
  stat[((size_t)w * EGG_STAT + 10 + c) * n + b] = u[((size_t)w * n + b) * 6 + c];
}

// The configurable MPC cost (egg_set_cost): one warp per world, lane l takes bodies l, l + 32, ...
// in that order and a fixed shuffle tree sums the lanes, so the summation order depends only on n:
// a world's cost has the same bits in any batch, shard or launch shape.
__device__ inline double egg_warp_sum(double s) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o);
  return s;
}

// sum_c q[c] d[c]^2 + l[c] d[c] over the 18 state components of body b, d = x - x_ref ([c][n] arrays)
__device__ inline double egg_state_cost(const double* x, const double* xr, const double* q, const double* l, int n, int b) {
  double s = 0.0;
#pragma unroll
  for (int c = 0; c < EGG_DYN; c++) {
    const double d = x[c * n + b] - xr[c * n + b];
    s += (q[c * n + b] * d + l[c * n + b]) * d;
  }
  return s;
}

// egg_fext_slice_kernel fused with the running cost of step t: the same f_ext writes, and
// cost[w] (= at t = 0, += after) the running term at (x_t, u_t), read in the same pass.  Left alone,
// ptxas hoists all 84 loads of a body and takes 255 registers with spills; the bound caps it at 64.
__global__ void __launch_bounds__(256, 4) egg_fext_slice_cost_kernel(const double* __restrict__ u, int W, int n, double* __restrict__ stat,
                                           const double* __restrict__ dyn, EggCost cc, const double* __restrict__ xr,
                                           int t, double* __restrict__ cost) {
  const long long w = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (w >= W) return;   // uniform over the warp
  const int lane = threadIdx.x & 31;
  const double* x = dyn + (size_t)w * EGG_DYN * n;
  double* f = stat + ((size_t)w * EGG_STAT + 10) * n;
  double s = 0.0;
#pragma unroll 1
  for (int b = lane; b < n; b += 32) {
    const double* ub = u + ((size_t)w * n + b) * 6;
    double r = egg_state_cost(x, xr, cc.q_run, cc.l_run, n, b);
#pragma unroll
    for (int j = 0; j < 6; j++) {
      const double uj = ub[j];
      f[j * n + b] = uj;
      r += cc.u_run[j * n + b] * uj * uj;
    }
    s += r;
  }
  s = egg_warp_sum(s);
  if (lane == 0) cost[w] = (t == 0) ? s : cost[w] + s;
}

// Actuator mode (egg_set_actuators): the f_ext slot of every body from a control row u [W][m] of
// actuator values, f = (m_b g, sum of +-tau_a over the actuators that touch b, in actuator order) with
// tau_a = u_a k_a, k_a = axis[a] or R(frame[a]) axis[a] from the state x_t.  Every product and sum is
// rounded on its own (no contraction), so the numpy transcription mpc.Actuators.wrench has the same
// bits.  One warp per world: lanes take bodies l, l + 32, ... and gather over the body's list, so no
// atomics.  With kCost the same pass adds the running cost of step t: the state part of
// egg_fext_slice_cost_kernel over the lane's bodies, then u_run[a] u_a^2 over actuators l, l + 32,
// ..., then the warp tree, so a world's J has the same bits in any batch.
template <bool kCost>
__global__ void __launch_bounds__(256, 4) egg_actuate_kernel(const double* __restrict__ u, int W, int n, double* __restrict__ stat,
                                                             const double* __restrict__ dyn, const double* __restrict__ bpar,
                                                             double g0, double g1, double g2, EggAct act, EggCost cc,
                                                             const double* __restrict__ xr, int t, double* __restrict__ cost) {
  const long long w = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (w >= W) return;   // uniform over the warp
  const int lane = threadIdx.x & 31;
  const double* x = dyn + (size_t)w * EGG_DYN * n;
  const double* uw = u + (size_t)w * act.m;
  const double* mass = bpar + ((size_t)w * EGG_BPAR + 3) * n;
  double* f = stat + ((size_t)w * EGG_STAT + 10) * n;
  double s = 0.0;
#pragma unroll 1
  for (int b = lane; b < n; b += 32) {
    const double mb = mass[b];
    double tx = 0.0, ty = 0.0, tz = 0.0;
#pragma unroll 1
    for (int i = act.start[b]; i < act.start[b + 1]; i++) {
      const int e = act.list[i], a = e >= 0 ? e : ~e;
      const int fr = act.frame[a];
      const double ua = uw[a];
      double kx = act.axis[3 * a], ky = act.axis[3 * a + 1], kz = act.axis[3 * a + 2];
      if (fr >= 0) {
        double R[9];
#pragma unroll
        for (int c = 0; c < 9; c++) R[c] = x[(3 + c) * n + fr];
        const double rx = __dadd_rn(__dadd_rn(__dmul_rn(R[0], kx), __dmul_rn(R[1], ky)), __dmul_rn(R[2], kz));
        const double ry = __dadd_rn(__dadd_rn(__dmul_rn(R[3], kx), __dmul_rn(R[4], ky)), __dmul_rn(R[5], kz));
        const double rz = __dadd_rn(__dadd_rn(__dmul_rn(R[6], kx), __dmul_rn(R[7], ky)), __dmul_rn(R[8], kz));
        kx = rx, ky = ry, kz = rz;
      }
      const double ax = __dmul_rn(ua, kx), ay = __dmul_rn(ua, ky), az = __dmul_rn(ua, kz);
      if (e >= 0) tx = __dadd_rn(tx, ax), ty = __dadd_rn(ty, ay), tz = __dadd_rn(tz, az);
      else tx = __dsub_rn(tx, ax), ty = __dsub_rn(ty, ay), tz = __dsub_rn(tz, az);
    }
    f[0 * n + b] = __dmul_rn(mb, g0);
    f[1 * n + b] = __dmul_rn(mb, g1);
    f[2 * n + b] = __dmul_rn(mb, g2);
    f[3 * n + b] = tx;
    f[4 * n + b] = ty;
    f[5 * n + b] = tz;
    if constexpr (kCost) s += egg_state_cost(x, xr, cc.q_run, cc.l_run, n, b);
  }
  if constexpr (kCost) {
#pragma unroll 1
    for (int a = lane; a < act.m; a += 32) {
      const double ua = uw[a];
      s += cc.u_run[a] * ua * ua;
    }
    s = egg_warp_sum(s);
    if (lane == 0) cost[w] = (t == 0) ? s : cost[w] + s;
  }
}

// The terminal term at x_H: cost[w] += sum_b sum_c q_term d^2 + l_term d.
__global__ void egg_cost_terminal_kernel(int W, int n, const double* __restrict__ dyn, EggCost cc,
                                         const double* __restrict__ xr, double* __restrict__ cost) {
  const long long w = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (w >= W) return;
  const int lane = threadIdx.x & 31;
  const double* x = dyn + (size_t)w * EGG_DYN * n;
  double s = 0.0;
#pragma unroll 1
  for (int b = lane; b < n; b += 32) s += egg_state_cost(x, xr, cc.q_term, cc.l_term, n, b);
  s = egg_warp_sum(s);
  if (lane == 0) cost[w] += s;
}

// The unpack kernel with a world-index map: dyn [W][18][n] of worlds[i] -> AoS out [k][n][18], the
// per-body order of egg_get_bodies (p, R row-major, v, w).
__global__ void egg_gather_state_kernel(const double* dyn, int n, const int* worlds, int k, double* out) {
  const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (gid >= (long long)k * n * EGG_DYN) return;
  const int c = (int)(gid % EGG_DYN);
  const long long t = gid / EGG_DYN;
  const int b = (int)(t % n);
  const int i = (int)(t / n);
  out[gid] = dyn[((size_t)worlds[i] * EGG_DYN + c) * n + b];
}

// AoS in [k][n][18] -> dyn of every world, world w from source (first + w) mod k.  One thread per
// (w, component, body) with the body fastest: the W x 18 x n writes are coalesced, the k x n x 18
// reads are small and stay in L2.
__global__ void egg_seed_state_kernel(double* dyn, int W, int n, const double* in, int k, int first) {
  const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (gid >= (long long)W * EGG_DYN * n) return;
  const int b = (int)(gid % n);
  const long long t = gid / n;
  const int c = (int)(t % EGG_DYN);
  const long long w = t / EGG_DYN;
  const long long src = ((long long)first + w) % k;
  dyn[gid] = in[((size_t)src * n + b) * EGG_DYN + c];
}

// FP64 roofline probe: 8 independent DFMA chains per thread.
__global__ void egg_dfma_kernel(double* out, int iters) {
  double a0 = threadIdx.x * 1e-3, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
  const double m = 1.0000001, c = 1e-7;
  for (int i = 0; i < iters; i++) {
    a0 = fma(a0, m, c); a1 = fma(a1, m, c); a2 = fma(a2, m, c); a3 = fma(a3, m, c);
    a4 = fma(a4, m, c); a5 = fma(a5, m, c); a6 = fma(a6, m, c); a7 = fma(a7, m, c);
  }
  double s = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
  if (s == 123.456) out[0] = s;
}

}  // namespace

double egg_measure_fp64_tflops() {
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  double* out = nullptr;
  if (cudaMalloc(&out, 8) != cudaSuccess) return -2.0;
  const int iters = 20000, threads = 256, blocks = sms * 8;
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0); cudaEventCreate(&e1);
  egg_dfma_kernel<<<blocks, threads>>>(out, 1000);
  double best = 0;
  for (int rep = 0; rep < 3; rep++) {
    cudaEventRecord(e0);
    egg_dfma_kernel<<<blocks, threads>>>(out, iters);
    cudaEventRecord(e1);
    cudaEventSynchronize(e1);
    float ms = 0;
    cudaEventElapsedTime(&ms, e0, e1);
    double tf = 2.0 * 8.0 * iters * (double)threads * blocks / (ms * 1e-3) / 1e12;
    if (tf > best) best = tf;
  }
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  cudaFree(out);
  return best;
}

cudaError_t egg_launch_init(const EggDev& d, cudaStream_t s) {
  long long t = (long long)d.W * d.n;
  cudaError_t e = cudaMemsetAsync(d.iso_flag, 0xff, sizeof(int), s);   // all ones; bit 0 cleared by a non-isotropic body, bit 1 by a non-uniform one
  egg_init_kernel<<<(unsigned)((t + 127) / 128), 128, 0, s>>>(d);
  egg_iso_uniform_kernel<<<(unsigned)((t + 127) / 128), 128, 0, s>>>(d);
  if (d.nj > 0) {
    long long tj = (long long)d.W * d.nj;
    egg_init_check_kernel<<<(unsigned)((tj + 127) / 128), 128, 0, s>>>(d);
  }
  EGG_FIRST(e, cudaGetLastError());
  return e;
}

cudaError_t egg_launch_clear_contacts(const EggDev& d, cudaStream_t s) {
  egg_clear_contacts_kernel<<<(d.W + 127) / 128, 128, 0, s>>>(d);
  return cudaGetLastError();
}

cudaError_t egg_launch_costs(const EggDev& d, double* cost_d, cudaStream_t s) {
  egg_cost_kernel<<<(d.W + 127) / 128, 128, 0, s>>>(d, cost_d);
  return cudaGetLastError();
}

cudaError_t egg_launch_pack(int W, const double* aos, int per_world, int comps, double* soa, int soa_comps, int comp_off, cudaStream_t s) {
  long long total = (long long)W * per_world * comps;
  if (total == 0) return cudaSuccess;
  egg_pack_kernel<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(aos, W, per_world, comps, soa, soa_comps, comp_off);
  return cudaGetLastError();
}
cudaError_t egg_launch_unpack(int W, double* aos, int per_world, int comps, const double* soa, int soa_comps, int comp_off, cudaStream_t s) {
  long long total = (long long)W * per_world * comps;
  if (total == 0) return cudaSuccess;
  egg_unpack_kernel<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(aos, W, per_world, comps, soa, soa_comps, comp_off);
  return cudaGetLastError();
}

cudaError_t egg_launch_fext_slice(const EggDev& d, const double* u, cudaStream_t s) {
  const long long total = (long long)d.W * 6 * d.n;
  egg_fext_slice_kernel<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(u, d.W, d.n, d.stat);
  return cudaGetLastError();
}
// x_ref row of step t (row 0 for a constant reference)
static const double* cost_ref_row(const EggDev& d, const EggCost& c, int t) {
  return c.x_ref + (size_t)(c.ref_steps == 1 ? 0 : t) * EGG_DYN * d.n;
}
cudaError_t egg_launch_fext_slice_cost(const EggDev& d, const double* u, const EggCost& c, int t, double* cost, cudaStream_t s) {
  const long long threads = (long long)d.W * 32;   // one warp per world
  egg_fext_slice_cost_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, s>>>(u, d.W, d.n, d.stat, d.dyn, c, cost_ref_row(d, c, t), t, cost);
  return cudaGetLastError();
}
cudaError_t egg_launch_actuate(const EggDev& d, const EggAct& a, const double* u, const EggCost* c, int t, double* cost, cudaStream_t s) {
  const long long threads = (long long)d.W * 32;   // one warp per world
  const unsigned blocks = (unsigned)((threads + 255) / 256);
  if (c)
    egg_actuate_kernel<true><<<blocks, 256, 0, s>>>(u, d.W, d.n, d.stat, d.dyn, d.bpar, d.prm.g[0], d.prm.g[1], d.prm.g[2], a, *c,
                                                    cost_ref_row(d, *c, t), t, cost);
  else
    egg_actuate_kernel<false><<<blocks, 256, 0, s>>>(u, d.W, d.n, d.stat, d.dyn, d.bpar, d.prm.g[0], d.prm.g[1], d.prm.g[2], a,
                                                     EggCost{}, nullptr, t, nullptr);
  return cudaGetLastError();
}
cudaError_t egg_launch_cost_terminal(const EggDev& d, const EggCost& c, int horizon, double* cost, cudaStream_t s) {
  const long long threads = (long long)d.W * 32;
  egg_cost_terminal_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, s>>>(d.W, d.n, d.dyn, c, cost_ref_row(d, c, horizon), cost);
  return cudaGetLastError();
}
cudaError_t egg_launch_gather_state(const EggDev& d, const int* worlds, int k, double* out, cudaStream_t s) {
  const long long total = (long long)k * d.n * EGG_DYN;
  egg_gather_state_kernel<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(d.dyn, d.n, worlds, k, out);
  return cudaGetLastError();
}
cudaError_t egg_launch_seed_state(const EggDev& d, const double* in, int k, int first, cudaStream_t s) {
  const long long total = (long long)d.W * EGG_DYN * d.n;
  egg_seed_state_kernel<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(d.dyn, d.W, d.n, in, k, first);
  return cudaGetLastError();
}
