// Matrix-free Jacobi and backward-SOR solvers (the other two members of the reference's
// sparse::*Iteration family), wired into the same ComputeVDot slot as the PGS kernel.
//
// Replaces (per world): sparse::JacobiIteration / SORIteration(constraints, M^-1, rhs, cfm)
// (/root/reference/eggshell/sparse_iterations.cc:148-226,269-286) with
// MatrixSolveSparseDiagonal / MatrixSolveSparseUpperTriangle and CalculateSparseLxUx / LxDx
// (/root/reference/eggshell/sparse_iterations_utils.cc:67-108,292-373,427-603), omega = 1.5.
//
// These are the reference's test-only solvers; the kernel is correctness-first: one warp per
// world, Jacobi's gather pass and the residual are lane-parallel, the order-dependent parts (SOR's
// reverse sweep, the re-accumulation of a = M^-1 J^T x) are walked by one lane in reference order.
// Same compact records and body structs as egg_pgs.cu.
#include "egg_internal.cuh"

namespace {

constexpr int BS = 17;   // per-body struct: a(6) | 1/m | I^-1(9), odd stride
constexpr double kSOR = 1.0 / 1.5;

struct Rec {
  double Rc[9];
  d3 r0, r1;
  double doff[3], ddiag[3], inva[3], rhs[3];
  int i0, i1, orig;
};
__device__ inline void load(const double* recs, int slot, Rec& r) {
  const double* f = recs + (size_t)slot * EGG_REC;
  for (int k = 0; k < 9; k++) r.Rc[k] = f[REC_RC + k];
  r.r0 = mk3(f[REC_R0], f[REC_R0 + 1], f[REC_R0 + 2]);
  r.r1 = mk3(f[REC_R1], f[REC_R1 + 1], f[REC_R1 + 2]);
  for (int k = 0; k < 3; k++) { r.doff[k] = f[REC_DOFF + k]; r.ddiag[k] = f[REC_DDIAG + k]; r.inva[k] = f[REC_INVA + k]; r.rhs[k] = f[REC_RHS + k]; }
  r.i0 = __double2loint(f[REC_IDX]); r.i1 = __double2hiint(f[REC_IDX]);
  r.orig = __double2loint(f[REC_META]);
}
__device__ inline d3 Ja(const Rec& r, const double* sb) {
  d3 u = mk3(0, 0, 0);
  if (r.i1 >= 0) { const double* q = sb + r.i1 * BS; u = mk3(q[0], q[1], q[2]) + cross3(mk3(q[3], q[4], q[5]), r.r1); }
  if (r.i0 >= 0) { const double* q = sb + r.i0 * BS; u = u - (mk3(q[0], q[1], q[2]) + cross3(mk3(q[3], q[4], q[5]), r.r0)); }
  return mmulv(r.Rc, u);
}
__device__ inline void scatter(const Rec& r, d3 delta, double* sb) {
  d3 imp = mtmulv(r.Rc, delta);
  if (r.i1 >= 0) {
    double* q = sb + r.i1 * BS;
    d3 da = mmulv(q + 7, cross3(r.r1, imp));
    q[0] += q[6] * imp.x; q[1] += q[6] * imp.y; q[2] += q[6] * imp.z; q[3] += da.x; q[4] += da.y; q[5] += da.z;
  }
  if (r.i0 >= 0) {
    double* q = sb + r.i0 * BS;
    d3 da = mmulv(q + 7, cross3(r.r0, imp));
    q[0] -= q[6] * imp.x; q[1] -= q[6] * imp.y; q[2] -= q[6] * imp.z; q[3] -= da.x; q[4] -= da.y; q[5] -= da.z;
  }
}
__device__ inline double clampk(double x, bool contact, int row) {   // ApplyProjection with the BOX bounds
  if (contact) {
    if (row < 2) { if (x < -1.0) return -1.0; else if (x > 1.0) return 1.0; }
    else if (x < 0.0) return 0.0;
  }
  return x;
}

__global__ void __launch_bounds__(32) egg_iter_kernel(EggDev d, double dt, int solver) {
  extern __shared__ double sb[];
  const int n = d.n, nj = d.nj, lane = threadIdx.x;
  const double cfm = d.prm.cfm, tol = d.prm.tol;
  const bool shift = (d.prm.quirks & 1) != 0;
  for (int w = blockIdx.x; w < d.W; w += gridDim.x) {
    const double* st = d.stat + (size_t)w * EGG_STAT * n;
    for (int i = lane; i < n * BS; i += 32) { const int b = i / BS, f = i - b * BS; sb[i] = (f >= 6 && f < 16) ? st[(f - 6) * n + b] : 0.0; }
    const int nc = nj + d.c_count[w];
    const double* recs = d.rec + (size_t)w * d.nrec * EGG_REC;
    const int* slot_of = d.slot_of + (size_t)w * d.nrec;
    double* x = d.lam + (size_t)w * d.nrec * 3;      // indexed by slot
    double* xn = d.lam2 + (size_t)w * d.nrec * 3;
    __syncwarp();
    // x0 = rhs; a = M^-1 J^T x0 accumulated in reference order
    for (int s = lane; s < nc; s += 32) { Rec r; load(recs, s, r); x[3 * s] = r.rhs[0]; x[3 * s + 1] = r.rhs[1]; x[3 * s + 2] = r.rhs[2]; }
    __syncwarp();
    auto rebuild_a = [&](const double* xv) {
      for (int i = lane; i < n * BS; i += 32) if (i % BS < 6) sb[i] = 0.0;
      __syncwarp();
      if (lane == 0)
        for (int c = 0; c < nc; c++) { Rec r; const int s = slot_of[c]; load(recs, s, r); scatter(r, mk3(xv[3 * s], xv[3 * s + 1], xv[3 * s + 2]), sb); }
      __syncwarp();
    };
    auto residual = [&](const double* xv) -> double {
      double se = 0, s1 = 0, s2 = 0, s3 = 0;
      for (int s = lane; s < nc; s += 32) {
        Rec r; load(recs, s, r);
        d3 t = Ja(r, sb);
        const bool eq = r.orig < nj;
        for (int k = 0; k < 3; k++) {
          const double xx = xv[3 * s + k], wv = get3(t, k) + cfm * xx - r.rhs[k];
          if (eq) { se += wv * wv; continue; }
          const double lo = (k < 2) ? -1.0 : 0.0;
          if (xx == lo && wv < 0) s1 += wv * wv;
          if (k < 2 && xx == 1.0 && wv > 0) s2 += wv * wv;
          if (xx > lo && (k == 2 || xx < 1.0)) s3 += wv * wv;
        }
      }
      for (int o = 16; o > 0; o >>= 1) {
        se += __shfl_xor_sync(0xffffffffu, se, o); s1 += __shfl_xor_sync(0xffffffffu, s1, o);
        s2 += __shfl_xor_sync(0xffffffffu, s2, o); s3 += __shfl_xor_sync(0xffffffffu, s3, o);
      }
      return sqrt(se) + (sqrt(s1) + sqrt(s2) + sqrt(s3));
    };
    double err = 0.0;
    int it = 0;
    if (nc > 0) {
      rebuild_a(x);
      err = residual(x);
      while (err > tol && it < d.prm.k_max) {
        if (solver == 2) {
          // Jacobi: x_k <- P((rhs_k - sum_{l != k} A_kl x_l) / (A_kk)), own bounds (MatrixSolveSparseDiagonal)
          for (int s = lane; s < nc; s += 32) {
            Rec r; load(recs, s, r);
            d3 t = Ja(r, sb);
            const bool contact = r.orig >= nj;
            for (int k = 0; k < 3; k++) {
              const double xo = x[3 * s + k];
              xn[3 * s + k] = clampk((r.rhs[k] - (get3(t, k) - r.ddiag[k] * xo)) * r.inva[k], contact, k);
            }
          }
          __syncwarp();
          for (int i = lane; i < 3 * nc; i += 32) x[i] = xn[i];
          __syncwarp();
          rebuild_a(x);
        } else {
          // backward SOR: blocks and rows descending, diagonal scaled by kSOR = 1/omega
          // (MatrixSolveSparseUpperTriangle with N = L + (1 - kSOR) D); q2: block i is projected
          // with the bounds of block i+1 (sparse_iterations_utils.cc:302,315,362-368).
          if (lane == 0) {
            for (int c = nc - 1; c >= 0; c--) {
              Rec r; const int s = slot_of[c]; load(recs, s, r);
              const int src = (shift && c + 1 < nc) ? c + 1 : c;
              const bool contact = src >= nj;
              d3 t = Ja(r, sb);
              double tt[3] = {t.x, t.y, t.z}, dl[3] = {0, 0, 0};
              // D(k,l) for l > k
              const double D01 = r.doff[0], D02 = r.doff[1], D12 = r.doff[2];
              for (int k = 2; k >= 0; k--) {
                double tk = tt[k];
                if (k == 1) tk += D12 * dl[2];
                if (k == 0) tk += D01 * dl[1] + D02 * dl[2];
                const double xo = x[3 * s + k], akk = r.ddiag[k] + cfm;
                const double num = r.rhs[k] - (tk - r.ddiag[k] * xo) - (1.0 - kSOR) * akk * xo - cfm * 0.0;
                // note: sum_{l != k} A_kl x_l excludes the cfm term of the diagonal; the (1-kSOR)
                // relaxation term carries (D_kk + cfm) as CalculateSparseDx does
                const double xnew = clampk(num / (kSOR * akk), contact, k);
                dl[k] = xnew - xo;
                x[3 * s + k] = xnew;
              }
              scatter(r, mk3(dl[0], dl[1], dl[2]), sb);
            }
          }
          __syncwarp();
        }
        err = residual(x);
        ++it;
      }
    }
    // outputs
    double* lo_out = d.lam_out + (size_t)w * 3 * d.nrec;
    int* rs_out = d.row_state + (size_t)w * 3 * d.nrec;
    for (int s = lane; s < nc; s += 32) {
      const int orig = __double2loint(recs[(size_t)s * EGG_REC + REC_META]);
      for (int k = 0; k < 3; k++) {
        const double xx = x[3 * s + k];
        lo_out[3 * orig + k] = xx;
        int state = 0;
        if (orig < nj) state = 3;
        else if (xx == ((k < 2) ? -1.0 : 0.0)) state = 1;
        else if (k < 2 && xx == 1.0) state = 2;
        rs_out[3 * orig + k] = state;
      }
    }
    if (lane == 0) {
      int* stt = d.stats + (size_t)w * 8;
      stt[4] = it; stt[5] = 0; stt[6] = (nc > 0 && cfm != 0.0); stt[7] = 0;   // no rows: ComputeVDot is never reached
      d.resid[w] = err;
    }
    // integrate: v' = v + dt (M^-1 f + a) etc. (ensembles.cc:535,572-591)
    double* dyn = d.dyn + (size_t)w * EGG_DYN * n;
    for (int b = lane; b < n; b += 32) {
      const double* q = sb + b * BS;
      d3 fl = mk3(st[10 * n + b], st[11 * n + b], st[12 * n + b]);
      d3 ft = mk3(st[13 * n + b], st[14 * n + b], st[15 * n + b]);
      d3 v = mk3(dyn[12 * n + b], dyn[13 * n + b], dyn[14 * n + b]);
      d3 wv = mk3(dyn[15 * n + b], dyn[16 * n + b], dyn[17 * n + b]);
      d3 vn = v + dt * (fl * q[6] + mk3(q[0], q[1], q[2]));
      d3 wn = wv + dt * (mmulv(q + 7, ft) + mk3(q[3], q[4], q[5]));
      d3 vmid = (v + vn) / 2.0, wmid = (wv + wn) / 2.0;
      d3 p = mk3(dyn[b], dyn[n + b], dyn[2 * n + b]) + dt * vmid;
      double z2 = dot3(wmid, wmid);
      d3 axis = (z2 > 0) ? wmid / sqrt(z2) : wmid;
      double ha = 0.5 * (norm3(wmid) * dt);
      double qw = cos(ha), sn = sin(ha);
      double qx = sn * axis.x, qy = sn * axis.y, qz = sn * axis.z;
      double tx = 2 * qx, ty = 2 * qy, tz = 2 * qz, twx = tx * qw, twy = ty * qw, twz = tz * qw;
      double txx = tx * qx, txy = ty * qx, txz = tz * qx, tyy = ty * qy, tyz = tz * qy, tzz = tz * qz;
      double Q[9] = {1 - (tyy + tzz), txy - twz, txz + twy, txy + twz, 1 - (txx + tzz), tyz - twx, txz - twy, tyz + twx, 1 - (txx + tyy)};
      double R[9], Rn[9];
      for (int k = 0; k < 9; k++) R[k] = dyn[(3 + k) * n + b];
      mmulm(Q, R, Rn);
      dyn[b] = p.x; dyn[n + b] = p.y; dyn[2 * n + b] = p.z;
      for (int k = 0; k < 9; k++) dyn[(3 + k) * n + b] = Rn[k];
      dyn[12 * n + b] = vn.x; dyn[13 * n + b] = vn.y; dyn[14 * n + b] = vn.z;
      dyn[15 * n + b] = wn.x; dyn[16 * n + b] = wn.y; dyn[17 * n + b] = wn.z;
      double chk = p.x + p.y + p.z + vn.x + vn.y + vn.z + wn.x + wn.y + wn.z;
      if (!(fabs(chk) < 1e300)) atomicOr(&d.status[w], 16);
    }
    __syncwarp();
  }
}

}  // namespace

size_t egg_iter_smem(const EggDev& d) { return (size_t)d.n * BS * sizeof(double); }

cudaError_t egg_launch_solve_iter(const EggDev& d, double dt, int solver, cudaStream_t s) {
  const size_t smem = egg_iter_smem(d);
  cudaError_t e = cudaSuccess;
  if (smem > 48 * 1024) {
    e = cudaFuncSetAttribute(egg_iter_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
  }
  int dev = 0, sms = 148;
  EGG_FIRST(e, cudaGetDevice(&dev));
  EGG_FIRST(e, cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  if (e != cudaSuccess) return e;
  int grid = d.W < sms * 16 ? d.W : sms * 16;
  egg_iter_kernel<<<grid, 32, smem, s>>>(d, dt, solver);
  return cudaGetLastError();
}
