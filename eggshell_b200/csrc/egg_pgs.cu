// Per-world constraint-row assembly and the dispatch of the PGS solver variants.
//
// Replaces (per world):
//   egg_assemble_kernel  Joint/Contact::ComputeJ + error  joints.cc:3-35, contact.cc:14-117,
//                        Ensemble::ComputeJ / rhs         ensembles.cc:38-87, 156-171, 563-570
// (record math in egg_record.cuh).  The per-world record layout written here feeds the dense path
// (egg_dense.cu), Jacobi / SOR (egg_iter.cu) and the position relaxation; the PGS kernel has its
// own group-stream assembly (egg_pgs_stream.cu).
//
// Formulation.  Every constraint (joint or contact) is one 3-row block whose two 3x6 Jacobians
// are [-Rc, Rc [r0]x] and [Rc, -Rc [r1]x] (contact.cc:60-75; a ball joint is the same shape with
// Rc = -I, joints.cc:22-30).  Instead of 2x3x6 Jacobian entries per block the kernels keep a
// compact 240-byte record (Rc, r0, r1, the 3x3 diagonal block D of J M^-1 J^T, rhs) and the
// body-space accumulator a = M^-1 J^T x (6 doubles per body, in shared memory).
//
// Schedule.  Gauss-Seidel is sequential in constraint order, but blocks that share no body
// commute exactly.  Blocks are grouped into dependency levels (level(c) = 1 + max level of any
// earlier block sharing a body) and levels are cut into stages of <= cap blocks; running stage
// after stage with one lane per block is bit-identical to the sequential sweep.
#include "egg_internal.cuh"
#include "egg_record.cuh"

namespace {

// ---------------------------------------------------------------------------------------------
// Assembly: one CTA per world.  Thread 0 computes the dependency levels / stages from the body
// indices staged in shared memory; then one thread per constraint builds its record and writes
// it at its (stage, lane) position in piece-major order.
template <int NT>
__global__ void __launch_bounds__(NT) egg_assemble_kernel(EggDev d, double dt, int stage_cap) {
  extern __shared__ double sm[];
  const int n = d.n, nj = d.nj, w = blockIdx.x, tid = threadIdx.x;
  double* sdyn = sm;                         // [18][n]
  double* sst = sm + EGG_DYN * n;            // [16][n]
  double* su = sm + (EGG_DYN + EGG_STAT) * n;         // [6][n] u = v/dt + M^-1 f per body
  int* si0 = (int*)(su + 6 * n);                       // [nrec]
  int* si1 = si0 + d.nrec;                   // [nrec]
  int* slot = si1 + d.nrec;                  // [nrec] record slot of c
  int* lev = slot + d.nrec;                  // [nrec] dependency level of c
  int* lstart = lev + d.nrec;                // [nrec + 1] level counts -> running slot cursor
  int* lstage = lstart + d.nrec + 1;         // [nrec + 1] first stage of each level
  int* lfirst = lstage + d.nrec + 1;         // [nrec + 1] first slot of each level
  int* blast = lfirst + d.nrec + 1;          // [n] last level that touched the body
  const double* dyn = d.dyn + (size_t)w * EGG_DYN * n;
  const double* st = d.stat + (size_t)w * EGG_STAT * n;
  for (int i = tid; i < EGG_DYN * n; i += NT) sdyn[i] = dyn[i];
  for (int i = tid; i < EGG_STAT * n; i += NT) sst[i] = st[i];
  const int ncon = d.c_count[w];
  const int nc = nj + ncon;
  const int* c_i0 = d.c_i0 + (size_t)w * d.maxc;
  const int* c_i1 = d.c_i1 + (size_t)w * d.maxc;
  const double* geom = d.c_geom + (size_t)w * 7 * d.maxc;
  for (int c = tid; c < nc; c += NT) {
    if (c < nj) { si0[c] = d.j_i0[(size_t)w * nj + c]; si1[c] = d.j_i1[(size_t)w * nj + c]; }
    else { si0[c] = c_i0[c - nj]; si1[c] = c_i1[c - nj]; }
  }
  for (int b = tid; b < n; b += NT) blast[b] = -1;
  for (int c = tid; c <= nc; c += NT) lstart[c] = 0;
  __syncthreads();
  egg_body_u(n, sdyn, sst, dt, su, tid, NT);

  int* gstage = d.level_start ? d.level_start + (size_t)w * (d.nrec + 1) : nullptr;
  if (tid == 0) {
    int nl = 0;
    for (int c = 0; c < nc; c++) {           // reference order: joints, then contacts
      const int i0 = si0[c], i1 = si1[c];
      int l = -1;
      if (i0 >= 0) l = max(l, blast[i0]);
      if (i1 >= 0) l = max(l, blast[i1]);
      l += 1;
      if (i0 >= 0) blast[i0] = l;
      if (i1 >= 0) blast[i1] = l;
      lev[c] = l;
      lstart[l]++;
      nl = max(nl, l + 1);
    }
    int ns = 0, run = 0;
    for (int l = 0; l < nl; l++) {
      const int cnt = lstart[l];
      lfirst[l] = run;
      lstart[l] = run;                       // running cursor of the level
      lstage[l] = ns;
      for (int k = 0; k < cnt; k += stage_cap) { if (gstage) gstage[ns] = run + k; ns++; }
      run += cnt;
    }
    if (gstage) gstage[ns] = nc;
    d.n_levels[w] = ns;
    for (int c = 0; c < nc; c++) slot[c] = lstart[lev[c]]++;   // stable inside a level
  }
  __syncthreads();

  double* recw = d.rec + (size_t)w * d.nrec * EGG_REC;
  for (int c = tid; c < nc; c += NT) {
    const int i0 = si0[c], i1 = si1[c];
    double v[EGG_REC];
    egg_build_record(d, w, c, i0, i1, sdyn, sst, su, geom, dt, false, v);
    if (d.slot_of) d.slot_of[(size_t)w * d.nrec + c] = slot[c];
    double2* out = reinterpret_cast<double2*>(recw + (size_t)slot[c] * EGG_REC);
#pragma unroll
    for (int p = 0; p < EGG_PIECES; p++) out[p] = make_double2(v[2 * p], v[2 * p + 1]);
  }
}

int g_num_sms = 0;
int num_sms() {
  if (!g_num_sms) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev);
    if (g_num_sms <= 0) g_num_sms = 148;
  }
  return g_num_sms;
}
bool stream_variant(const EggDev& d) { return d.rec_fmt != 0; }

}  // namespace

// Lanes per world of the PGS kernel = maximum blocks per stage the assembly may emit.  The
// overrides come from d.sel (read by egg_create).
int egg_stage_cap(const EggDev& d) {
  int lpw = d.sel.lpw;
  if (stream_variant(d)) {
    // narrow worlds expose little parallelism per level: fewer lanes, more worlds per warp
    // (measured: stack10 87 ms at 1 / 101 at 2 / 133 at 4; legged20 95 ms at 4 / 115 at 2 / 123 at 8)
    // -- unless the batch is too small to give every SM a few warps that way
    if (lpw != 1 && lpw != 2 && lpw != 4 && lpw != 8 && lpw != 16) {
      lpw = (d.n <= 12) ? 1 : (d.n <= 24 ? 4 : 8);
      const long long want = (long long)num_sms() * d.sel.min_warps;
      while (lpw < 8 && (long long)d.W * lpw / 32 < want) lpw *= 2;
    }
    return lpw;
  }
  return 8;   // per-world records (dense, Jacobi / SOR, relaxation): the stage cut is not used by those kernels
}

size_t egg_assemble_smem(const EggDev& d) {
  return (size_t)(EGG_DYN + EGG_STAT + 6) * d.n * sizeof(double) + (size_t)(7 * d.nrec + d.n + 8) * sizeof(int);
}

int egg_assemble_threads(const EggDev& d) {
  if (d.rec_fmt) return egg_records_threads(d);
  return d.nrec <= 128 ? 64 : 256;
}

cudaError_t egg_launch_assemble(const EggDev& d, double dt, cudaStream_t s) {
  if (d.rec_fmt) return egg_launch_assemble_stream(d, dt, s);
  const size_t smem = egg_assemble_smem(d);
  const int cap = egg_stage_cap(d);
  cudaError_t e = cudaSuccess;
  if (egg_assemble_threads(d) == 64) {
    if (smem > 48 * 1024) e = cudaFuncSetAttribute(egg_assemble_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    egg_assemble_kernel<64><<<d.W, 64, smem, s>>>(d, dt, cap);
  } else {
    if (smem > 48 * 1024) e = cudaFuncSetAttribute(egg_assemble_kernel<256>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    egg_assemble_kernel<256><<<d.W, 256, smem, s>>>(d, dt, cap);
  }
  return cudaGetLastError();
}

cudaError_t egg_launch_solve_pgs(const EggDev& d, double dt, const double* mu, cudaStream_t s) { return egg_launch_solve_pgs_stream(d, dt, mu, s); }
