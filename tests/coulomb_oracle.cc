// TEST INFRASTRUCTURE ONLY: the Coulomb-pyramid friction of egg_set_friction on the CPU oracle.
//
// Built by tests/coulomb_oracle.py with the flags of oracle/Makefile (no FMA contraction) and loaded
// next to oracle/liboracle.so.  It includes the oracle's unchanged headers and steps a World created
// by liboracle.so (same header, same flags: the same layout), so everything the oracle does besides
// the Gauss-Seidel solve -- narrowphase, de-duplication, rows, rhs, integration -- is the oracle's own
// code.  What differs from orc::sparse_iteration / orc::sparse_solve_lower (INTEGRATION.md,
// "Friction"):
//   * sweep k -> k+1 bounds block i's tangent rows, when the block is projected as a contact (with
//     q2 the kind comes from its neighbour), by [-b, b], b = mu max(x_n, 0), x_n = block i's normal
//     multiplier in x_k;
//   * each update records per tangent row a clamp flag (0 free, 1 at -b, 2 at +b; 0 for rows not
//     projected as a contact and for x_0), which the residual and row_state read for the tangent
//     rows of contact blocks instead of comparing x with a constant.
#include <map>
#include "../oracle/orc_world.h"

using namespace orc;

namespace {

struct Cone {
  double mu;
  std::vector<unsigned char> flag;   // per row
  Vec bound;                         // per row: b of the last projection as a contact (inf: none)
};

// orc::sparse_solve_lower (eps = cfm, scale = 1) with the cone; xk is the iterate the sweep starts from.
Vec solve_lower_cone(const BlockSystem& B, const Vec& rhs, double eps, bool quirk, Cone& cone, const Vec& xk) {
  Vec x(B.nc * 3, 0.0);
  const double inf = std::numeric_limits<double>::infinity();
  for (int i = 0; i < B.nc; i++) {
    double sub[3] = {0, 0, 0};
    for (int e = B.start[i]; e < B.start[i + 1]; e++) {
      int j = B.col[e];
      if (j > i) break;
      for (int r = 0; r < 3; r++) {
        double s = 0;
        for (int c = 0; c < 3; c++) s += B.blk[(size_t)e * 9 + r * 3 + c] * x[3 * j + c];
        sub[r] += s;
      }
    }
    double d[3][3];
    for (int r = 0; r < 3; r++) for (int c = 0; c < 3; c++) d[r][c] = B.diag[(size_t)i * 9 + r * 3 + c] + (r == c ? eps : 0.0);
    const int src = bounds_source(i, B.nc, true, quirk);
    for (int k = 0; k < 3; k++) {
      for (int l = 0; l < k; l++) sub[k] += d[k][l] * x[3 * i + l];
      const double v = (rhs[3 * i + k] - sub[k]) / d[k][k];
      double lo = B.lo[3 * src + k], hi = B.hi[3 * src + k];
      if (k < 2) {
        const bool proj = !B.type[3 * src + k];
        double b = inf;
        if (proj) {
          const double xn = xk[3 * i + 2];
          b = cone.mu * (xn > 0.0 ? xn : 0.0);
          lo = -b; hi = b;
        }
        cone.flag[3 * i + k] = !proj ? 0 : (v < lo ? 1 : (v > hi ? 2 : 0));
        cone.bound[3 * i + k] = b;
      }
      x[3 * i + k] = apply_projection(v, B.type[3 * src + k], lo, hi);
    }
  }
  return x;
}

// orc::residual_error with the tangent rows of contact blocks judged by their clamp flags.
double residual_cone(const Vec& w, const Vec& x, const std::vector<unsigned char>& C, const Vec& lo, const Vec& hi,
                     const std::vector<unsigned char>& flag) {
  double se = 0, s1 = 0, s2 = 0, s3 = 0;
  for (size_t i = 0; i < w.size(); i++) {
    if (C[i]) { se += w[i] * w[i]; continue; }
    if (i % 3 < 2) {
      if (flag[i] == 1 && w[i] < 0) s1 += w[i] * w[i];
      if (flag[i] == 2 && w[i] > 0) s2 += w[i] * w[i];
      if (flag[i] == 0) s3 += w[i] * w[i];
      continue;
    }
    if (x[i] == lo[i] && w[i] < 0) s1 += w[i] * w[i];
    if (x[i] == hi[i] && w[i] > 0) s2 += w[i] * w[i];
    if (x[i] > lo[i] && x[i] < hi[i]) s3 += w[i] * w[i];
  }
  return std::sqrt(se) + (std::sqrt(s1) + std::sqrt(s2) + std::sqrt(s3));
}

// orc::sparse_iteration, Gauss-Seidel, with the cone.
Vec gs_iteration_cone(const BlockSystem& B, const Vec& rhs, double cfm, int k_max, double tol, bool quirk, Cone& cone,
                      int* sweeps_out, double* resid_out) {
  Vec x = rhs;
  int it = 0;
  if (B.nc == 0) { *sweeps_out = 0; *resid_out = 0; return Vec(); }
  auto resid = [&](const Vec& xx) {
    Vec w = sparse_Ax(B, xx, cfm);
    for (size_t i = 0; i < w.size(); i++) w[i] -= rhs[i];
    return residual_cone(w, xx, B.type, B.lo, B.hi, cone.flag);
  };
  double err = resid(x);
  while (err > tol && it < k_max) {
    Vec nx = sparse_Ux(B, x);
    Vec irhs(nx.size());
    for (size_t i = 0; i < nx.size(); i++) irhs[i] = -1 * nx[i] + rhs[i];
    x = solve_lower_cone(B, irhs, cfm, quirk, cone, x);
    err = resid(x);
    ++it;
  }
  *sweeps_out = it;
  *resid_out = err;
  return x;
}

// orc::world_step on the PGS path with the cone (the other solvers have no Coulomb friction).
void world_step_cone(World& W, double dt, double mu, Vec* bound_out) {
  const int n = W.n;
  W.stats.status &= ~ST_LCP_FAILED;
  Vec v(6 * n);
  for (int i = 0; i < n; i++) {
    v[6 * i + 0] = W.bodies[i].v.x; v[6 * i + 1] = W.bodies[i].v.y; v[6 * i + 2] = W.bodies[i].v.z;
    v[6 * i + 3] = W.bodies[i].w.x; v[6 * i + 4] = W.bodies[i].w.y; v[6 * i + 5] = W.bodies[i].w.z;
  }
  update_contacts(W);
  check_and_correct(W);
  std::vector<Rows3> rows;
  all_rows(W, &rows);
  const int nr = (int)rows.size() * 3;
  W.stats.n_rows = nr;
  W.stats.sweeps = W.stats.pivots = W.stats.cfm_applied = 0;
  W.stats.residual = 0;
  Vec err = position_error(W);
  Vec u(6 * n);
  for (int i = 0; i < n; i++) {
    for (int k = 0; k < 3; k++) u[6 * i + k] = v[6 * i + k] / dt + W.Minv_lin[i] * W.f_ext[6 * i + k];
    Vec3 t = W.Minv_ang[i] * Vec3(W.f_ext[6 * i + 3], W.f_ext[6 * i + 4], W.f_ext[6 * i + 5]);
    for (int k = 0; k < 3; k++) u[6 * i + 3 + k] = v[6 * i + 3 + k] / dt + t[k];
  }
  Vec rhs(nr);
  for (size_t c = 0; c < rows.size(); c++)
    for (int r = 0; r < 3; r++) {
      double s = 0;
      if (rows[c].i0 >= 0) for (int k = 0; k < 6; k++) s += rows[c].j0[r][k] * u[6 * rows[c].i0 + k];
      if (rows[c].i1 >= 0) for (int k = 0; k < 6; k++) s += rows[c].j1[r][k] * u[6 * rows[c].i1 + k];
      rhs[3 * c + r] = -W.prm.erp / dt / dt * err[3 * c + r] - s;
    }
  W.rhs = rhs;
  Vec lambda(nr, 0.0);
  W.row_state.assign(nr, 0);
  Cone cone{mu, std::vector<unsigned char>(nr, 0), Vec(nr, std::numeric_limits<double>::infinity())};
  if (nr > 0) {
    BlockSystem B;
    build_block_system(W, &B);
    lambda = gs_iteration_cone(B, rhs, W.prm.cfm, W.prm.k_max, W.prm.tol, (W.prm.quirks & QUIRK_GS_BOUNDS_SHIFT) != 0, cone,
                               &W.stats.sweeps, &W.stats.residual);
    W.stats.cfm_applied = W.prm.cfm != 0;
    for (int i = 0; i < nr; i++) {
      if (B.type[i]) W.row_state[i] = 3;
      else if (i % 3 < 2) W.row_state[i] = cone.flag[i];
      else if (lambda[i] == B.lo[i]) W.row_state[i] = 1;
      else if (lambda[i] == B.hi[i]) W.row_state[i] = 2;
      else W.row_state[i] = 0;
    }
  }
  W.lambda = lambda;
  *bound_out = cone.bound;
  Vec g = W.f_ext;
  for (size_t c = 0; c < rows.size(); c++)
    for (int r = 0; r < 3; r++) {
      double l = lambda[3 * c + r];
      if (rows[c].i0 >= 0) for (int k = 0; k < 6; k++) g[6 * rows[c].i0 + k] += rows[c].j0[r][k] * l;
      if (rows[c].i1 >= 0) for (int k = 0; k < 6; k++) g[6 * rows[c].i1 + k] += rows[c].j1[r][k] * l;
    }
  Vec vn(6 * n);
  for (int i = 0; i < n; i++) {
    for (int k = 0; k < 3; k++) vn[6 * i + k] = v[6 * i + k] + dt * (W.Minv_lin[i] * g[6 * i + k]);
    Vec3 t = W.Minv_ang[i] * Vec3(g[6 * i + 3], g[6 * i + 4], g[6 * i + 5]);
    for (int k = 0; k < 3; k++) vn[6 * i + 3 + k] = v[6 * i + 3 + k] + dt * t[k];
  }
  for (int i = 0; i < n; i++) {
    Body& b = W.bodies[i];
    b.v = Vec3(vn[6 * i], vn[6 * i + 1], vn[6 * i + 2]);
    b.w = Vec3(vn[6 * i + 3], vn[6 * i + 4], vn[6 * i + 5]);
    Vec3 vmid = (Vec3(v[6 * i], v[6 * i + 1], v[6 * i + 2]) + b.v) / 2.0;
    b.p = b.p + dt * vmid;
    Vec3 wmid = (Vec3(v[6 * i + 3], v[6 * i + 4], v[6 * i + 5]) + b.w) / 2.0;
    b.R = quat_to_mat(w_to_q(wmid, dt)) * b.R;
  }
}

std::map<const void*, Vec> g_bound;   // per world: the bound tap of its last Coulomb step

}  // namespace

extern "C" {

// One step of the world at wp (an orc_world_create handle) with Coulomb friction mu (finite, >= 0).
// Returns the status word, or -1 (nothing stepped) for a bad mu or a solver other than PGS.
int coulomb_world_step(void* wp, double dt, double mu) {
  World& W = *(World*)wp;
  if (!std::isfinite(mu) || mu < 0 || W.prm.solver != SOLVER_PGS) return -1;
  world_step_cone(W, dt, mu + 0.0, &g_bound[wp]);   // + 0.0: -0.0 becomes +0.0, as egg_set_friction stores it
  return W.stats.status;
}
// The bound each row was last projected with in the world's last Coulomb step (inf: none); returns its length.
int coulomb_world_bound(void* wp, double* out) {
  const Vec& b = g_bound[wp];
  if (out) std::copy(b.begin(), b.end(), out);
  return (int)b.size();
}
void coulomb_world_forget(void* wp) { g_bound.erase(wp); }

}  // extern "C"
