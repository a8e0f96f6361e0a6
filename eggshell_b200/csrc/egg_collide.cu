// Narrowphase kernel: box-ground + all-pairs box-box SAT / manifold with ordered compaction and
// the pair-local part of the reference's constraint de-duplication.
//
// Replaces (per world): Ensemble::UpdateContacts (/root/reference/eggshell/ensembles.cc:445-480),
// CollideBoxAndGround / CollideBoxes (/root/reference/eggshell/collision.cc:408-432, 166-388 with
// helpers :47,:70,:84,:105) and Ensemble::CheckAndCorrectEnsembleState (ensembles.cc:241-388).
//
// One CTA per world.  The world's p and R (12 n doubles) are staged in shared memory; SAT runs
// uniformly over all n(n-1)/2 pairs, colliding pairs are compacted IN ORDER with a block scan,
// and only the compacted list runs the divergent clipping code.  Contacts are written at
// prefix-sum slots so the list order equals the reference's (ground contacts body by body in
// vertex order, then pairs (i<j) lexicographic, each in emission order) without atomics.
//
// This translation unit is compiled with -fmad=false: every comparison against a threshold
// (collision.cc:189-190,218,249,282,369,419) must see exactly the value the FP64 CPU arithmetic
// produces, because hit / code / count are compared bit-exactly with the oracle.
#include "egg_internal.cuh"
#include <cstdlib>
#include <cfloat>

namespace {

struct BoxD {
  d3 c;
  double R[9];
  d3 h;
};

struct Sat {
  double R[9];   // box2 in box1's frame
  d3 p;
  int aacount;
  double mFN, mEE;
  d3 aFN, aEE;   // aEE in box1's frame
  int cFN, cEE;
};

// collision.cc:192-271.  Returns false as soon as one axis separates.
__device__ bool sat_test(const BoxD& b1, const BoxD& b2, Sat& s) {
  const double kAlignmentTolerance = 0.9962;
  const double kTolerance = 1e-9;
  const double* R1 = b1.R;
  const double* R2 = b2.R;
  // R = R1^T R2
  for (int i = 0; i < 3; i++)
    for (int j = 0; j < 3; j++) s.R[3 * i + j] = R1[i] * R2[j] + R1[3 + i] * R2[3 + j] + R1[6 + i] * R2[6 + j];
  s.p = mtmulv(R1, b2.c - b1.c);
  double Q[9];
  for (int k = 0; k < 9; k++) Q[k] = fabs(s.R[k]);
  s.aacount = 0;
  for (int i = 0; i < 3; i++) {
    double mx = fmax(Q[i], fmax(Q[3 + i], Q[6 + i]));
    s.aacount += (mx > kAlignmentTolerance);
  }
  const d3 H1 = b1.h, H2 = b2.h;
  s.mFN = -DBL_MAX;
  s.cFN = 0;
  s.aFN = mk3(0, 0, 0);
#pragma unroll
  for (int i = 0; i < 3; i++) {
    double e1 = get3(s.p, i);
    double separation = fabs(e1) - (get3(H1, i) + dot3(H2, mrow(Q, i)));
    if (separation > 0) return false;
    if (separation > s.mFN) { s.mFN = separation; s.aFN = sign1(e1) * mcol(R1, i); s.cFN = 1 + i; }
  }
#pragma unroll
  for (int i = 0; i < 3; i++) {
    double e1 = dot3(mcol(s.R, i), s.p);
    double separation = fabs(e1) - (dot3(H1, mcol(Q, i)) + get3(H2, i));
    if (separation > 0) return false;
    if (separation > s.mFN) { s.mFN = separation; s.aFN = sign1(e1) * mcol(R2, i); s.cFN = 4 + i; }
  }
  s.mEE = -DBL_MAX;
  s.cEE = 0;
  s.aEE = mk3(0, 0, 0);
#pragma unroll
  for (int i = 0; i < 3; i++) {
    const int i1 = (i + 1) % 3, i2 = (i + 2) % 3;
    const int ia = (i == 0) ? 1 : 0, ib = (i == 2) ? 1 : 2;
#pragma unroll
    for (int j = 0; j < 3; j++) {
      const int ja = (j == 0) ? 1 : 0, jb = (j == 2) ? 1 : 2;
      d3 nn = mk3(0, 0, 0);
      set3(nn, i1, -s.R[3 * i2 + j]);
      set3(nn, i2, s.R[3 * i1 + j]);
      double len = norm3(nn);
      if (!(len > kTolerance)) continue;
      double e1 = get3(s.p, i2) * s.R[3 * i1 + j] - get3(s.p, i1) * s.R[3 * i2 + j];
      double extent = get3(H1, ia) * Q[3 * ib + j] + get3(H1, ib) * Q[3 * ia + j] +
                      get3(H2, ja) * Q[3 * i + jb] + get3(H2, jb) * Q[3 * i + ja];
      double separation = fabs(e1) - extent;
      if (separation > 0) return false;
      separation /= len;
      if (separation > s.mEE) { s.mEE = separation; s.aEE = nn / (sign1(e1) * len); s.cEE = 7 + 3 * i + j; }
    }
  }
  return true;
}

// The same 15 axis tests when only the verdict "collide or not" is wanted (phase 1: collision.cc:218,249
// return false on the first positive separation): no normalisation, no tracking of the deepest
// axis.  An edge axis is skipped when its length is <= 1e-9 (collision.cc:240): the length is only
// compared with the threshold, so the square root is taken only when the squared length is
// within a hair of 1e-18 (the comparison on the root is then evaluated exactly as in sat_test).
__device__ bool sat_hits(const BoxD& b1, const BoxD& b2) {
  const double kTolerance = 1e-9;
  const double* R1 = b1.R;
  const double* R2 = b2.R;
  double R[9], Q[9];
  for (int i = 0; i < 3; i++)
    for (int j = 0; j < 3; j++) R[3 * i + j] = R1[i] * R2[j] + R1[3 + i] * R2[3 + j] + R1[6 + i] * R2[6 + j];
  const d3 p = mtmulv(R1, b2.c - b1.c);
  for (int k = 0; k < 9; k++) Q[k] = fabs(R[k]);
  const d3 H1 = b1.h, H2 = b2.h;
#pragma unroll
  for (int i = 0; i < 3; i++) {
    const double separation = fabs(get3(p, i)) - (get3(H1, i) + dot3(H2, mrow(Q, i)));
    if (separation > 0) return false;
  }
#pragma unroll
  for (int i = 0; i < 3; i++) {
    const double e1 = dot3(mcol(R, i), p);
    const double separation = fabs(e1) - (dot3(H1, mcol(Q, i)) + get3(H2, i));
    if (separation > 0) return false;
  }
#pragma unroll
  for (int i = 0; i < 3; i++) {
    const int i1 = (i + 1) % 3, i2 = (i + 2) % 3;
    const int ia = (i == 0) ? 1 : 0, ib = (i == 2) ? 1 : 2;
#pragma unroll
    for (int j = 0; j < 3; j++) {
      const int ja = (j == 0) ? 1 : 0, jb = (j == 2) ? 1 : 2;
      d3 nn = mk3(0, 0, 0);
      set3(nn, i1, -R[3 * i2 + j]);
      set3(nn, i2, R[3 * i1 + j]);
      const double l2 = dot3(nn, nn);
      if (l2 < 0.99e-18) continue;                               // len <= 1e-9 for certain
      if (l2 < 1.01e-18 && !(sqrt(l2) > kTolerance)) continue;   // borderline: the reference's own test
      const double e1 = get3(p, i2) * R[3 * i1 + j] - get3(p, i1) * R[3 * i2 + j];
      const double extent = get3(H1, ia) * Q[3 * ib + j] + get3(H1, ib) * Q[3 * ia + j] +
                            get3(H2, ja) * Q[3 * i + jb] + get3(H2, jb) * Q[3 * i + ja];
      if (fabs(e1) - extent > 0) return false;
    }
  }
  return true;
}

// norm3(v) < dmin without the square root unless |v|^2 is within a hair of dmin^2.
__device__ __forceinline__ bool closer_than(d3 v, double dmin) {
  const double d2 = dot3(v, v), t2 = dmin * dmin;
  if (d2 > t2 * 1.000001) return false;
  if (d2 < t2 * 0.999999) return dmin > 0;
  return sqrt(d2) < dmin;
}

// collision.cc:47-62
__device__ void line_closest_approach(d3 pa, d3 ua, d3 pb, d3 ub, double* alpha, double* beta) {
  d3 p = pb - pa;
  double uaub = dot3(ua, ub);
  double q1 = dot3(ua, p);
  double q2 = -dot3(ub, p);
  double d = 1 - uaub * uaub;
  if (d == 0) { *alpha = 0; *beta = 0; }
  else { *alpha = (q1 + uaub * q2) / d; *beta = (uaub * q1 + q2) / d; }
}

// collision.cc:84-99 with :70-80 inlined.  Returns the new vertex count.
__device__ int clip_polygon(const double* px, const double* py, int np, double nx, double ny, double d,
                            double* ox, double* oy) {
  int m = 0;
  for (int i = 0; i < np; i++) {
    int i2 = (i + 1 == np) ? 0 : i + 1;
    double k1 = nx * px[i] + ny * py[i] + d;
    if (k1 >= 0 && m < EGG_MAX_POLY) { ox[m] = px[i]; oy[m] = py[i]; m++; }
    double k2 = nx * px[i2] + ny * py[i2] + d;
    if (k1 * k2 < 0 && m < EGG_MAX_POLY) {
      double t = k1 / (k2 - k1);
      ox[m] = px[i] - t * (px[i2] - px[i]);
      oy[m] = py[i] - t * (py[i2] - py[i]);
      m++;
    }
  }
  return m;
}

// collision.cc:273-388 (everything after the 15 axis tests).  out: [k][4] = pos, depth; every contact of
// a manifold carries the same normal (*nrm_out), so the per-thread contact buffer holds it once.
__device__ int manifold(const BoxD& box1, const BoxD& box2, const Sat& s, int* code_out, double* out, d3* nrm_out) {
  const double kTolerance = 1e-9;
  const double* R1 = box1.R;
  const double* R2 = box2.R;
  d3 aEE = mmulv(R1, s.aEE);
  bool best_FN = (s.mFN > s.mEE);
  if (s.aacount == 0 && !best_FN) {
    *code_out = s.cEE;
    d3 pa = box1.c, pb = box2.c;
#pragma unroll
    for (int j = 0; j < 3; j++) {
      pa = pa + (sign1(dot3(aEE, mcol(R1, j))) * get3(box1.h, j)) * mcol(R1, j);
      pb = pb - (sign1(dot3(aEE, mcol(R2, j))) * get3(box2.h, j)) * mcol(R2, j);
    }
    d3 ua = mcol(R1, (s.cEE - 7) / 3);
    d3 ub = mcol(R2, (s.cEE - 7) % 3);
    double alpha, beta;
    line_closest_approach(pa, ua, pb, ub, &alpha, &beta);
    d3 pos = (pa + ua * alpha + pb + ub * beta) * 0.5;
    out[0] = pos.x; out[1] = pos.y; out[2] = pos.z;
    out[3] = -s.mEE;
    *nrm_out = aEE;
    return 1;
  }
  *code_out = s.cFN;
  const bool first = (s.cFN <= 3);
  const BoxD& A = first ? box1 : box2;
  const BoxD& Bo = first ? box2 : box1;
  d3 Aface_normal = s.aFN * (first ? 1.0 : -1.0);
  d3 nf = mtmulv(Bo.R, Aface_normal);
  int nfi = 0;
  {
    double best = fabs(nf.x);
    if (fabs(nf.y) > best) { best = fabs(nf.y); nfi = 1; }
    if (fabs(nf.z) > best) { best = fabs(nf.z); nfi = 2; }
  }
  d3 Bface_normal = (-sign1(get3(nf, nfi))) * mcol(Bo.R, nfi);
  // Incident face rectangle: centre, two in-plane axes, plane normal, half sides.
  d3 Rc = Bo.c + Bface_normal * get3(Bo.h, nfi);
  d3 Rx = mcol(Bo.R, (nfi + 1) % 3), Ry = mcol(Bo.R, (nfi + 2) % 3), Rn = mcol(Bo.R, nfi);
  double hx = get3(Bo.h, (nfi + 1) % 3), hy = get3(Bo.h, (nfi + 2) % 3);
  d3 AfaceCenter = A.c + Aface_normal * get3(A.h, (s.cFN - 1) % 3);
  double Ad = -dot3(Aface_normal, AfaceCenter);

  // collision.cc:105-158 IntersectBoxAndRectangle(A, rect)
  double px[EGG_MAX_POLY], py[EGG_MAX_POLY], qx[EGG_MAX_POLY], qy[EGG_MAX_POLY];
  int np = 4;
  px[0] = -hx; py[0] = -hy;
  px[1] = -hx; py[1] = hy;
  px[2] = hx;  py[2] = hy;
  px[3] = hx;  py[3] = -hy;
  d3 Bc = A.c - Rc;
  bool cur_is_p = true;
  for (int i = 0; i < 3 && np > 0; i++) {
    d3 Bnormal = mcol(A.R, i);
    double BnBc = dot3(Bnormal, Bc);
    double crs = norm3(cross3(Bnormal, Rn));
    for (int j = -1; j <= 1 && np > 0; j += 2) {
      double Bd = (double)(-j) * BnBc - get3(A.h, i);
      if (crs < kTolerance) {
        if (Bd <= 0) continue;
        np = 0;
        break;
      }
      double Hx = dot3(Rx, Bnormal), Hy = dot3(Ry, Bnormal);
      if (cur_is_p) np = clip_polygon(px, py, np, (double)(-j) * Hx, (double)(-j) * Hy, -Bd, qx, qy);
      else np = clip_polygon(qx, qy, np, (double)(-j) * Hx, (double)(-j) * Hy, -Bd, px, py);
      cur_is_p = !cur_is_p;
    }
  }
  const double* fx = cur_is_p ? px : qx;
  const double* fy = cur_is_p ? py : qy;
  int cnt = 0;
  for (int i = 0; i < np; i++) {
    d3 pos = Rc + Rx * fx[i] + Ry * fy[i];
    double depth = -(dot3(Aface_normal, pos) + Ad);
    if ((fabs(depth) > kTolerance || s.aacount >= 2) && cnt < EGG_MAX_PAIR_CONTACTS) {
      double* o = out + 4 * cnt;
      o[0] = pos.x; o[1] = pos.y; o[2] = pos.z;
      o[3] = depth;
      cnt++;
    }
  }
  if (cnt == 0) {
    out[0] = box2.c.x; out[1] = box2.c.y; out[2] = box2.c.z;
    out[3] = -s.mFN;
    *code_out = 16;
    cnt = 1;
  }
  *nrm_out = s.aFN;
  return cnt;
}

template <int NT>
__device__ int block_excl_scan(int v, int* total, int* wsum) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  int inc = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    int t = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += t;
  }
  if (NT == 32) {     // one warp per world: the warp scan is the block scan (no barrier, no shared memory)
    *total = __shfl_sync(0xffffffffu, inc, 31);
    return inc - v;
  }
  __syncthreads();   // protects wsum reuse across consecutive calls
  if (lane == 31) wsum[wid] = inc;
  __syncthreads();
  int base = 0, tot = 0;
#pragma unroll
  for (int k = 0; k < NT / 32; k++) {
    int sv = wsum[k];
    if (k < wid) base += sv;
    tot += sv;
  }
  *total = tot;
  return base + inc - v;
}

__device__ inline void pair_from_index(int q, int n, int* pi, int* pj) {
  // q = i (2n - i - 1)/2 + (j - i - 1)
  const float tn = 2.0f * (float)n - 1.0f;           // a float estimate is enough: the two loops below make it exact
  int i = (int)floorf((tn - sqrtf(tn * tn - 8.0f * (float)q)) * 0.5f);
  if (i < 0) i = 0;
  while (i > 0 && (i * (2 * n - i - 1)) / 2 > q) i--;
  while (((i + 1) * (2 * n - i - 2)) / 2 <= q) i++;
  *pi = i;
  *pj = q - (i * (2 * n - i - 1)) / 2 + i + 1;
}

__device__ inline void load_box(const double* sp, const double* sR, const double* side, int n, int b, BoxD& box) {
  box.c = mk3(sp[b], sp[n + b], sp[2 * n + b]);
#pragma unroll
  for (int k = 0; k < 9; k++) box.R[k] = sR[k * n + b];
  box.h = mk3(side[b] * 0.5, side[n + b] * 0.5, side[2 * n + b] * 0.5);
}

template <int NT>
__global__ void __launch_bounds__(NT) egg_collide_kernel(EggDev d) {
  extern __shared__ double sm[];
  const int n = d.n, P = d.P, w = blockIdx.x, tid = threadIdx.x;
  double* sp = sm;                 // [3][n]
  double* sR = sm + 3 * n;         // [9][n]
  double* sside = sm + 12 * n;     // [3][n]
  double* srad = sm + 15 * n;      // [n] bounding-sphere radius
  double* sshape = sm + 16 * n;    // [n] collider: 0 box, 1 sphere, 2 capsule (sside = its dims)
  unsigned short* hitlist = (unsigned short*)(sm + 17 * n);          // [P] cull survivors, then colliding pairs
  unsigned char* hit = (unsigned char*)(hitlist + ((P + 3) & ~3));   // [P]
  __shared__ int wsum[NT / 32];
  __shared__ int s_flags;

  const double* dyn = d.dyn + (size_t)w * EGG_DYN * n;
  const double* bpar = d.bpar + (size_t)w * EGG_BPAR * n;
  for (int i = tid; i < 12 * n; i += NT) sm[i] = dyn[i];
  for (int i = tid; i < 3 * n; i += NT) sside[i] = bpar[i];
  for (int i = tid; i < n; i += NT) sshape[i] = bpar[13 * n + i];
  if (tid == 0) s_flags = 0;
  __syncthreads();
  for (int b = tid; b < n; b += NT) {
    const int shp = (int)sshape[b];
    srad[b] = (shp == 0) ? norm3(mk3(sside[b] * 0.5, sside[n + b] * 0.5, sside[2 * n + b] * 0.5))
                         : (shp == 1 ? sside[b] : sside[n + b] * 0.5 + sside[b]);
  }

  int* c_i0 = d.c_i0 + (size_t)w * d.maxc;
  int* c_i1 = d.c_i1 + (size_t)w * d.maxc;
  int* c_code = d.c_code + (size_t)w * d.maxc;
  double* geom = d.c_geom + (size_t)w * 7 * d.maxc;
  const int maxc = d.maxc;

  // ---- box vs ground (collision.cc:408-432): vertex order x,y,z nested, contact iff v.z < 0 ----
  int base = 0, raw = 0;
  for (int b0 = 0; b0 < n; b0 += NT) {
    const int b = b0 + tid;
    unsigned mask = 0;
    d3 vert[8];
    if (b < n) {
      d3 c = mk3(sp[b], sp[n + b], sp[2 * n + b]);
      d3 c0 = mk3(sR[0 * n + b], sR[3 * n + b], sR[6 * n + b]);
      d3 c1 = mk3(sR[1 * n + b], sR[4 * n + b], sR[7 * n + b]);
      d3 c2 = mk3(sR[2 * n + b], sR[5 * n + b], sR[8 * n + b]);
      double s0 = sside[b], s1 = sside[n + b], s2 = sside[2 * n + b];
      const int shp = (int)sshape[b];
      if (shp == 0) {
        int k = 0;
        for (int x = -1; x <= 1; x += 2)
          for (int y = -1; y <= 1; y += 2)
            for (int z = -1; z <= 1; z += 2) {
              d3 v = c + c0 * s0 * 0.5 * (double)x + c1 * s1 * 0.5 * (double)y + c2 * s2 * 0.5 * (double)z;
              vert[k] = v;
              if (v.z < 0) mask |= 1u << k;
              k++;
            }
      } else {
        // sphere / capsule (oracle/orc_collision.h collide_round_and_ground): the lowest point of each
        // end sphere, -z end first; s0 = radius, s1 = axis length
        const int ends = (shp == 2) ? 2 : 1;
        for (int e = 0; e < ends; e++) {
          d3 ce = c;
          if (shp == 2) ce = c + c2 * (s1 * 0.5 * (e == 0 ? -1.0 : 1.0));
          d3 v = mk3(ce.x, ce.y, ce.z - s0);
          vert[e] = v;
          if (v.z < 0) mask |= 1u << e;
        }
      }
    }
    int cnt = __popc(mask), tot;
    int off = block_excl_scan<NT>(cnt, &tot, wsum);
    int slot = base + off;
    for (int k = 0; k < 8; k++)
      if (mask & (1u << k)) {
        if (slot < maxc) {
          c_i0[slot] = -1; c_i1[slot] = b; c_code[slot] = 0;
          geom[0 * maxc + slot] = vert[k].x; geom[1 * maxc + slot] = vert[k].y; geom[2 * maxc + slot] = vert[k].z;
          geom[3 * maxc + slot] = 0.0; geom[4 * maxc + slot] = 0.0; geom[5 * maxc + slot] = 1.0;
          geom[6 * maxc + slot] = -vert[k].z;
        }
        slot++;
      }
    base += tot;
  }
  raw = base;

  // ---- phase 1: cull, then SAT on the survivors; hit flags ----
  // Conservative cull in front of the SAT (SURVEY row f3; the reference's own broadphase,
  // toolkit/collision.cc:58-109, is unused by Ensemble::UpdateContacts): boxes whose bounding
  // spheres are apart by a 1e-3 relative margin are disjoint, so one of the 15 axes separates
  // them by a margin far above rounding and CollideBoxes returns false (collision.cc:218,249).
  // The colliding-pair list is unchanged (tests/test_gpu_parity.py::test_broadphase_cull_keeps_pair_list);
  // EGG_OPT_NO_BROADPHASE_CULL (quirks bit 8) runs the SAT on every pair.  The survivors are
  // compacted first (order irrelevant here) so that the SAT runs on full warps.
  __syncthreads();                 // srad
  int nsurv = 0;
  {
    const bool nocull = (d.prm.quirks & 8) != 0;
    for (int q0 = 0; q0 < P; q0 += NT) {
      const int q = q0 + tid;
      int keep = 0;
      if (q < P) {
        int i, j;
        pair_from_index(q, n, &i, &j);
        const d3 dc = mk3(sp[j] - sp[i], sp[n + j] - sp[n + i], sp[2 * n + j] - sp[2 * n + i]);
        const double rr = srad[i] + srad[j];
        keep = (nocull || !(dot3(dc, dc) > rr * rr * 1.002)) ? 1 : 0;
        hit[q] = 0;
        if (d.pair_code) { d.pair_code[(size_t)w * P + q] = 0; d.pair_cnt[(size_t)w * P + q] = 0; }
      }
      int tot;
      const int off = block_excl_scan<NT>(keep, &tot, wsum);
      if (keep) hitlist[nsurv + off] = (unsigned short)q;
      nsurv += tot;
    }
  }
  __syncthreads();
  for (int h = tid; h < nsurv; h += NT) {
    const int q = hitlist[h];
    int i, j;
    pair_from_index(q, n, &i, &j);
    const int s1 = (int)sshape[i], s2 = (int)sshape[j];
    if (s1 == 0 && s2 == 0) {
      BoxD b1, b2;
      load_box(sp, sR, sside, n, i, b1);
      load_box(sp, sR, sside, n, j, b2);
      if (sat_hits(b1, b2)) hit[q] = 1;
    } else if (s1 == 1 && s2 == 1) {          // sphere - sphere (oracle/orc_collision.h collide_spheres)
      const d3 dc = mk3(sp[j] - sp[i], sp[n + j] - sp[n + i], sp[2 * n + j] - sp[2 * n + i]);
      const double depth = (sside[i] + sside[j]) - norm3(dc);
      if (depth > 0) hit[q] = 1;
    }                                          // other collider pairs: no pairwise narrowphase
  }
  __syncthreads();

  // ---- ordered compaction of the hit pairs ----
  int nhits = 0;
  for (int q0 = 0; q0 < P; q0 += NT) {
    const int q = q0 + tid;
    int f = (q < P) ? hit[q] : 0, tot;
    int off = block_excl_scan<NT>(f, &tot, wsum);
    if (f) hitlist[nhits + off] = (unsigned short)q;
    nhits += tot;
  }
  __syncthreads();

  // ---- phase 2: manifolds + pair-local de-duplication on the compacted list ----
  const double dmin = d.prm.min_dist;
  const int nj = d.nj;
  const int* j_i0 = d.j_i0 + (size_t)w * nj;
  const int* j_i1 = d.j_i1 + (size_t)w * nj;
  const double* jc = d.jc + (size_t)w * 6 * nj;
  for (int h0 = 0; h0 < nhits; h0 += NT) {
    const int h = h0 + tid;
    double cb[4 * EGG_MAX_PAIR_CONTACTS];     // pos, depth per contact
    d3 cn = mk3(0, 0, 0);                      // the manifold's normal
    int cnt = 0, rawcnt = 0, code = 0, bi = 0, bj = 0;
    if (h < nhits) {
      const int q = hitlist[h];
      pair_from_index(q, n, &bi, &bj);
      BoxD b1, b2;
      load_box(sp, sR, sside, n, bi, b1);
      load_box(sp, sR, sside, n, bj, b2);
      if ((int)sshape[bi] == 1) {               // sphere - sphere: one contact in the middle of the overlap
        const d3 dc = b2.c - b1.c;
        const double dist = norm3(dc), r1 = sside[bi], r2 = sside[bj];
        const double depth = (r1 + r2) - dist;
        const d3 nn = (dist > 0) ? dc / dist : mk3(0, 0, 1);
        const d3 pos = b1.c + nn * (r1 - depth * 0.5);
        cb[0] = pos.x; cb[1] = pos.y; cb[2] = pos.z; cb[3] = depth;
        cn = nn;
        code = 17;
        rawcnt = 1;
      } else {
        Sat s;
        sat_test(b1, b2, s);
        rawcnt = manifold(b1, b2, s, &code, cb, &cn);
      }
      if (d.pair_code) { d.pair_code[(size_t)w * P + q] = (unsigned char)code; d.pair_cnt[(size_t)w * P + q] = (unsigned char)rawcnt; }
      // CheckAndCorrectEnsembleState, restricted to this body pair (ensembles.cc:264-313):
      // joint-contact closer than dmin => drop the contact; contact-contact => drop the later.
      unsigned del = 0;
      for (int k = 0; k < nj; k++) {
        int a0 = j_i0[k], a1 = j_i1[k];
        int lo = a0 < a1 ? a0 : a1, hi = a0 < a1 ? a1 : a0;
        if (lo != bi || hi != bj) continue;
        d3 ca = mk3(jc[0 * nj + k], jc[1 * nj + k], jc[2 * nj + k]);
        d3 cbv = mk3(jc[3 * nj + k], jc[4 * nj + k], jc[5 * nj + k]);
        BoxD& B0 = (a0 == bi) ? b1 : b2;
        BoxD& B1 = (a1 == bi) ? b1 : b2;
        d3 p0 = B0.c + mmulv(B0.R, ca);
        d3 p1 = B1.c + mmulv(B1.R, cbv);
        d3 jp = (p0 + p1) / 2.0;
        for (int c = 0; c < rawcnt; c++) {
          d3 cp = mk3(cb[4 * c], cb[4 * c + 1], cb[4 * c + 2]);
          if (closer_than(jp - cp, dmin)) del |= 1u << c;
        }
      }
      for (int a = 0; a < rawcnt; a++)
        for (int b = a + 1; b < rawcnt; b++) {
          d3 pa = mk3(cb[4 * a], cb[4 * a + 1], cb[4 * a + 2]);
          d3 pb = mk3(cb[4 * b], cb[4 * b + 1], cb[4 * b + 2]);
          if (closer_than(pa - pb, dmin)) del |= 1u << b;
        }
      for (int c = 0; c < rawcnt; c++)
        if (!(del & (1u << c))) {
          if (cnt != c)
            for (int k = 0; k < 4; k++) cb[4 * cnt + k] = cb[4 * c + k];
          cnt++;
        }
    }
    int tot, rtot;
    int off = block_excl_scan<NT>(cnt, &tot, wsum);
    block_excl_scan<NT>(rawcnt, &rtot, wsum);
    int slot = base + off;
    for (int c = 0; c < cnt; c++, slot++) {
      if (slot >= maxc) continue;
      c_i0[slot] = bi; c_i1[slot] = bj; c_code[slot] = code;
      geom[0 * maxc + slot] = cb[4 * c]; geom[1 * maxc + slot] = cb[4 * c + 1]; geom[2 * maxc + slot] = cb[4 * c + 2];
      geom[3 * maxc + slot] = cn.x; geom[4 * maxc + slot] = cn.y; geom[5 * maxc + slot] = cn.z;
      geom[6 * maxc + slot] = cb[4 * c + 3];
    }
    base += tot;
    raw += rtot;
  }

  // Joint-joint conflicts between the same two bodies (ensembles.cc:278-287 would Panic).
  for (int k = tid; k < nj; k += NT) {
    int a0 = j_i0[k], a1 = j_i1[k];
    int lo = a0 < a1 ? a0 : a1, hi = a0 < a1 ? a1 : a0;
    if (lo < 0) continue;
    for (int k2 = k + 1; k2 < nj; k2++) {
      int e0 = j_i0[k2], e1 = j_i1[k2];
      int lo2 = e0 < e1 ? e0 : e1, hi2 = e0 < e1 ? e1 : e0;
      if (lo2 != lo || hi2 != hi) continue;
      d3 pos[2];
      for (int t = 0; t < 2; t++) {
        int kk = t ? k2 : k, f0 = t ? e0 : a0, f1 = t ? e1 : a1;
        BoxD B0, B1;
        load_box(sp, sR, sside, n, f0, B0);
        load_box(sp, sR, sside, n, f1, B1);
        d3 q0 = B0.c + mmulv(B0.R, mk3(jc[0 * nj + kk], jc[1 * nj + kk], jc[2 * nj + kk]));
        d3 q1 = B1.c + mmulv(B1.R, mk3(jc[3 * nj + kk], jc[4 * nj + kk], jc[5 * nj + kk]));
        pos[t] = (q0 + q1) / 2.0;
      }
      if (norm3(pos[0] - pos[1]) < dmin) atomicOr(&s_flags, 2 /*EGG_ST_JOINT_CONFLICT*/);
    }
  }
  __syncthreads();
  if (tid == 0) {
    int flags = s_flags;
    int count = base;
    if (count > maxc) { count = maxc; flags |= 8 /*EGG_ST_CONTACT_OVERFLOW*/; }
    d.c_count[w] = count;
    // LCP_FAILED is per step; the other bits are sticky.
    d.status[w] = (d.status[w] & ~1) | flags;
    int* st = d.stats + (size_t)w * 8;
    st[0] = raw;
    st[1] = count;
    st[2] = 3 * (nj + count);
    st[3] = nhits;
  }
}

}  // namespace

size_t egg_collide_smem(const EggDev& d) { return (size_t)17 * d.n * sizeof(double) + (size_t)((d.P + 3) & ~3) * 2 + (size_t)((d.P + 7) & ~7); }

// Threads per world by its pair count: one warp for small worlds (every barrier and block scan
// is paid per warp).  Measured, 131072 x 20 bodies (190 pairs): 3.45 ms at 256 threads, 2.56 at
// 128, 1.52 at 64, 1.08 at 32; 16384 x 64 bodies (2016 pairs): 2.81 ms at 256, 3.41 at 128.
// EGG_COLLIDE_NT (d.sel.collide_nt) = 32 / 64 / 128 picks that instance, any other value 256.
int egg_collide_threads(const EggDev& d) {
  const int nt = d.sel.collide_nt ? d.sel.collide_nt : (d.P <= 256 ? 32 : (d.P <= 600 ? 64 : (d.P <= 1200 ? 128 : 256)));
  return (nt == 32 || nt == 64 || nt == 128) ? nt : 256;
}

cudaError_t egg_launch_collide(const EggDev& d, cudaStream_t s) {
  const size_t smem = egg_collide_smem(d);
  cudaError_t e = cudaSuccess;
  const int nt = egg_collide_threads(d);
  if (nt == 32) {
    egg_collide_kernel<32><<<d.W, 32, smem, s>>>(d);
  } else if (nt == 64) {
    egg_collide_kernel<64><<<d.W, 64, smem, s>>>(d);
  } else if (nt == 128) {
    egg_collide_kernel<128><<<d.W, 128, smem, s>>>(d);
  } else {
    static thread_local size_t attr_set = 0;       // the attribute only ever has to grow
    if (smem > 48 * 1024 && smem > attr_set) {
      e = cudaFuncSetAttribute(egg_collide_kernel<256>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      if (e != cudaSuccess) return e;
      attr_set = smem;
    }
    egg_collide_kernel<256><<<d.W, 256, smem, s>>>(d);
  }
  return cudaGetLastError();
}
