// Run format of the projected Gauss-Seidel solve (opt-in: EGG_OPT_PGS_RUNS; isotropic bodies, FP64 records).
//
// What the previous kernel (egg_pgs_stream.cu, one block per lane and stage) left on the table
// (profiles/r1i_pgs_stream_final_summary.txt, per-line stall samples): a warp-stage of ~2200
// cycles of which the block arithmetic is ~570; header decode, guards, prefetch cursor, copy issue
// and the wait for the copy are paid per STAGE, and the stage count is the dependency depth of the
// world (pile64: 121 levels for 495 blocks).  And 272 stream bytes per block pass (then; 240 since the
// third frame row is rebuilt and the packed word travels with the multipliers), 72 of them a
// contact frame that the contacts of one manifold share.
//
// Here the unit of scheduling is a RUN: up to RUN_MAX consecutive contacts of the reference order
// on the same ordered body pair with the same normal (a box-box manifold, ensembles.cc:449-473, or
// one body's ground contacts).  They would occupy consecutive dependency levels anyway; one lane
// carries both bodies' accumulators in registers through the run -- the same arithmetic in the
// same order as the sequential sweep -- so the level count drops (pile64 121 -> 76, stack10
// 54 -> 27) and the per-stage overhead is paid once per run.  The record shrinks to what cannot
// be rebuilt (layout in egg_stream.cuh): 64 B per run (frame quaternion, r1 - r0, body indices) +
// 80 B per block (r0, 1/(D+cfm), rhs) + the 32-byte multiplier sector: pile64 ~188 B per block
// pass instead of 272.  The frame matrix comes from the quaternion with the expressions of the
// assembly (egg_record.cuh), r1 = r0 + (r1 - r0 of the run's first block), and the off-diagonal of
// the block's D from  D = s I - c0 q0 q0^T - c1 q1 q1^T  (q = Rc r, c = 1/inertia; exact for the
// isotropic bodies this kernel is selected for) -- all off the dependent chain of the update.
//
// Everything else is the algorithm of egg_pgs_stream.cu: group stream (G = 32/LPW worlds per warp
// interleaved round by round, one bulk copy per warp-stage), probe-based stopping test (here the
// probe chunk is read with plain loads: no second barrier, no staging slices), increment-form row
// update, cross-proxy fence before the staging buffer goes back to the TMA unit, fused integrate.
//
// Replaces: sparse::GaussSeidelIteration + GetResidualError + the velocity/position update,
// sparse_iterations.cc:148-226,51-69, sparse_iterations_utils.cc:12-21,159-243,495-695,
// ensembles.cc:535,572-591; assembly: Ensemble::ComputeJ / rhs (ensembles.cc:38-87,156-171,563-570).
#include "egg_internal.cuh"
#include "egg_record.cuh"
#include "egg_stream.cuh"
#include <cstdlib>

namespace {

// bit positions of the packed words
constexpr unsigned BK_KIND = 20, BK_EQ = 21;     // multiplier sector, 4th double (low word: reference constraint index)
constexpr unsigned RK_JOINT = 20;                // run record

// ---------------------------------------------------------------------------------------------
// Assembly 2/3 (run format): round headers and byte offsets of one group (one warp per group).
__global__ void __launch_bounds__(128) egg_rounds_runs_kernel(EggDev d, int G) {
  const int g = blockIdx.x * 4 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  const int ngroups = (d.W + G - 1) / G;
  if (g >= ngroups) return;
  const int nrec = d.nrec, LPW = 32 / G;
  int R = 0;
  for (int s = 0; s < G; s++) { const int w = g * G + s; if (w < d.W) R = max(R, d.n_levels[w]); }
  unsigned char* gs = reinterpret_cast<unsigned char*>(d.rec) + (size_t)g * group_stride_bytes(nrec, G);
  unsigned* roff = d.round_off + (size_t)g * (nrec + 1);
  // run lengths of round t (4 bits per lane of the warp), its blocks and runs
  auto lens_of = [&](int t, unsigned* lens, int& total, int& nruns) {
    lens[0] = lens[1] = lens[2] = lens[3] = 0u;
    total = nruns = 0;
    for (int s = 0; s < G; s++) {
      const int w = g * G + s;
      if (w >= d.W || t >= d.n_levels[w]) continue;
      const unsigned r = d.st_runs[(size_t)w * nrec + t];
      const int l0 = s * LPW;
      lens[l0 >> 3] |= r << ((l0 & 7) * 4);
      for (int l = 0; l < LPW; l++) { const int L = (r >> (4 * l)) & 15; total += L; nruns += (L > 0); }
    }
  };
  unsigned base = 0;
  for (int t0 = 0; t0 < R; t0 += 32) {
    const int t = t0 + lane;
    unsigned lens[4] = {0, 0, 0, 0}, lensn[4];
    int total = 0, nruns = 0, totn = 0, nrn = 0;
    unsigned bytes = 0, bytes_next = 0;
    if (t < R) {
      lens_of(t, lens, total, nruns);
      lens_of((t + 1) % R, lensn, totn, nrn);
      bytes = runs_round_bytes(total, nruns);
      bytes_next = runs_round_bytes(totn, nrn);
    }
    unsigned incl = bytes;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const unsigned v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += v; }
    const unsigned off = base + incl - bytes;
    if (t < R) {
      roff[t] = off;
      uint4* hp = reinterpret_cast<uint4*>(gs + off);
      hp[0] = make_uint4(lens[0], lens[1], lens[2], lens[3]);
      hp[1] = make_uint4(bytes, bytes_next, (unsigned)total | ((unsigned)nruns << 16), 0u);
      hp[2] = make_uint4(0u, 0u, 0u, 0u);
      hp[3] = make_uint4(0u, 0u, 0u, 0u);
    }
    base += __shfl_sync(0xffffffffu, incl, 31);
  }
  if (lane == 0) {
    int* gi = d.grp_info + (size_t)g * 4;
    unsigned l0[4];
    int t0 = 0, r0 = 0;
    if (R > 0) lens_of(0, l0, t0, r0);
    gi[0] = R;
    gi[1] = (R > 0) ? (int)runs_round_bytes(t0, r0) : 0;     // bytes of round 0
    gi[2] = (int)base;                                        // bytes of the stream
    gi[3] = 0;
  }
}

// Position of (lane, k) inside a round from the header's run lengths: j0 = index of the lane's run
// among the runs (= of its k = 0 block), jk = index of its k-th block in the k-major block order.
__device__ __forceinline__ void run_slot(const uint4 lens, int lane, int k, int& j0, int& jk, int& total, int& nruns) {
  const unsigned w4[4] = {lens.x, lens.y, lens.z, lens.w};
  const int wi = lane >> 3;
  const unsigned below = (1u << ((lane & 7) * 4)) - 1u;
  total = 0; nruns = 0; j0 = 0; jk = 0;
#pragma unroll
  for (int kk = 0; kk < RUN_MAX; kk++) {
    int cnt = 0, rank = 0;
#pragma unroll
    for (int q = 0; q < 4; q++) {
      const unsigned m = nib_ge(w4[q], kk + 1);
      cnt += __popc(m);
      if (q < wi) rank += __popc(m);
      else if (q == wi) rank += __popc(m & below);
    }
    if (kk == 0) { nruns = cnt; j0 = rank; }
    if (kk == k) jk = total + rank;
    total += cnt;
  }
}

// Assembly 3/3 (run format): one CTA per world builds the records and writes them at their round positions.
template <int NT>
__global__ void __launch_bounds__(NT, (NT >= 256) ? 2 : 4) egg_records_runs_kernel(EggDev d, double dt, int G) {
  extern __shared__ double sm[];
  const int n = d.n, nj = d.nj, w = blockIdx.x, tid = threadIdx.x, nrec = d.nrec;
  double* sdyn = sm;                         // [18][n]
  double* sst = sm + EGG_DYN * n;            // [16][n]
  double* su = sst + EGG_STAT * n;           // [6][n] u = v/dt + M^-1 f per body
  const double* dyn = d.dyn + (size_t)w * EGG_DYN * n;
  const double* st = d.stat + (size_t)w * EGG_STAT * n;
  for (int i = tid; i < EGG_DYN * n; i += NT) sdyn[i] = dyn[i];
  for (int i = tid; i < EGG_STAT * n; i += NT) sst[i] = st[i];
  __syncthreads();
  egg_body_u(n, sdyn, sst, dt, su, tid, NT);
  __syncthreads();
  const int nc = nj + d.c_count[w];
  const int g = w / G, sub = w % G, LPW = 32 / G;
  const int* c_i0 = d.c_i0 + (size_t)w * d.maxc;
  const int* c_i1 = d.c_i1 + (size_t)w * d.maxc;
  const double* geom = d.c_geom + (size_t)w * 7 * d.maxc;
  const int* cp = d.c_pos + (size_t)w * nrec;
  const unsigned* roff = d.round_off + (size_t)g * (nrec + 1);
  unsigned char* gs = reinterpret_cast<unsigned char*>(d.rec) + (size_t)g * group_stride_bytes(nrec, G);
  for (int c = tid; c < nc; c += NT) {
    int i0, i1;
    if (c < nj) { i0 = d.j_i0[(size_t)w * nj + c]; i1 = d.j_i1[(size_t)w * nj + c]; }
    else { i0 = c_i0[c - nj]; i1 = c_i1[c - nj]; }
    double v[EGG_REC];
    egg_build_record(d, w, c, i0, i1, sdyn, sst, su, geom, dt, true, v);
    const int p = cp[c], stg = p >> 8, ln = (p >> 3) & 31, k = p & 7;
    const unsigned ro = roff[stg];
    const uint4 lens = *reinterpret_cast<const uint4*>(gs + ro);
    int j0, jk, total, nruns;
    run_slot(lens, sub * LPW + ln, k, j0, jk, total, nruns);
    const int ckind = __double2hiint(v[REC_META]);
    const unsigned long long pkb = (unsigned long long)c | ((unsigned long long)ckind << BK_KIND) | ((unsigned long long)(c < nj ? 1 : 0) << BK_EQ);
    unsigned char* lamp = gs + ro + HDRB;
    unsigned char* runp = lamp + (size_t)LAMB * total;
    unsigned char* blkp = runp + (size_t)RUNB * nruns;
    double2* lam = reinterpret_cast<double2*>(lamp + (size_t)LAMB * jk);
    lam[0] = make_double2(v[REC_RHS], v[REC_RHS + 1]);              // x0 = rhs
    lam[1] = make_double2(v[REC_RHS + 2], __longlong_as_double((long long)pkb));
    auto bcol = [&](int col) { return reinterpret_cast<double2*>(blkp + ((size_t)col * total + jk) * 16); };
    // The solve rebuilds r1 as r0 + (r1 - r0 of the run's first block): exact bookkeeping for two
    // bodies (both lever arms end at the same contact point).  A ground / anchor side has no lever
    // arm (everything it multiplies is zero): a contact stores the arm of its real body in the r0
    // slot and a zero offset.
    d3 r0s = mk3(v[REC_R0], v[REC_R0 + 1], v[REC_R0 + 2]);
    d3 dps = mk3(v[REC_R1] - v[REC_R0], v[REC_R1 + 1] - v[REC_R0 + 1], v[REC_R1 + 2] - v[REC_R0 + 2]);
    if (c >= nj && (i0 < 0 || i1 < 0)) {
      if (i0 < 0) r0s = mk3(v[REC_R1], v[REC_R1 + 1], v[REC_R1 + 2]);
      dps = mk3(0, 0, 0);
    }
    *bcol(0) = make_double2(r0s.x, r0s.y);
    *bcol(1) = make_double2(r0s.z, v[REC_INVA]);
    *bcol(2) = make_double2(v[REC_INVA + 1], v[REC_INVA + 2]);
    *bcol(3) = make_double2(v[REC_RHS], v[REC_RHS + 1]);
    *bcol(4) = make_double2(v[REC_RHS + 2], 0.0);
    if (k == 0) {
      double q[4] = {1.0, 0.0, 0.0, 0.0};        // joints: frame -I = -(identity rotation), flagged below
      if (c >= nj) {
        const int kc = c - nj;
        egg_align_quat(mk3(geom[3 * d.maxc + kc], geom[4 * d.maxc + kc], geom[5 * d.maxc + kc]), q);
      }
      const unsigned long long pkr = (unsigned long long)(i0 + 1) | ((unsigned long long)(i1 + 1) << 10) | ((unsigned long long)(c < nj ? 1 : 0) << RK_JOINT);
      auto rcol = [&](int col) { return reinterpret_cast<double2*>(runp + ((size_t)col * nruns + j0) * 16); };
      *rcol(0) = make_double2(q[0], q[1]);
      *rcol(1) = make_double2(q[2], q[3]);
      *rcol(2) = make_double2(dps.x, dps.y);
      *rcol(3) = make_double2(dps.z, __longlong_as_double((long long)pkr));
    }
  }
}

enum { MODE_INIT = 0, MODE_UPDATE = 1, MODE_RESID = 2 };
enum { PH_INIT = 0, PH_PROBE = 1, PH_EXACT = 2, PH_UPDATE = 3 };

// ISO == 1: every body's M^-1 is (1/m) I3, (1/c) I3 (one 16-byte load per body); ISO == 2: the same
// pair for every body of the batch (kernel constants).  General inertia: egg_pgs_stream.cu.
template <int LPW, int ISO>
__global__ void __launch_bounds__(32, 11) egg_pgs_runs_kernel(EggDev d, double dt, int pf, int stage_cap) {
  constexpr int G = 32 / LPW;
  constexpr int RM = RUN_MAX;
  extern __shared__ __align__(128) unsigned char smraw[];
  const int n = d.n, lane = threadIdx.x, sub = lane / LPW, sl = lane % LPW;
  // shared memory: [mbarrier 8 B][pad][dummy body 48 B at 16: the ground / world anchor, always zero]
  //                [G x n x 6 doubles accumulators at 64][staging: one round]
  const unsigned bar = s32(smraw);
  double* sb = reinterpret_cast<double*>(smraw + 64) + (size_t)sub * 6 * n;
  const int dummy = -(sub * n) - 1;            // body index of the dummy relative to this world's sb
  unsigned char* stage0 = smraw + 64 + (size_t)G * 48 * n;
  const unsigned stage_s = s32(stage0);
  const double cfm = d.prm.cfm;
  const int nj = d.nj;
  const unsigned FULL = 0xffffffffu;
  const unsigned lt = (1u << lane) - 1u;
  const unsigned wmask = (LPW == 32) ? FULL : (((1u << LPW) - 1u) << (sub * LPW));   // the lanes of this lane's world

  if (lane == 0) {
    mbar_init(bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (lane < 6) reinterpret_cast<double*>(smraw + 16)[lane] = 0.0;
  const unsigned long long pol = policy_evict_first();
  const unsigned long long pol_keep = policy_evict_last();
  double um = 0.0, uc = 0.0;                   // ISO == 2: the batch-wide (1/m, 1/c)
  if (ISO == 2) { um = d.minv_iso[0]; uc = d.minv_iso[1]; }
  __syncwarp();
  unsigned parity = 0;
  const int ngroups = (d.W + G - 1) / G;

  while (true) {
    int grp = 0;
    if (lane == 0) grp = atomicAdd(d.work_ctr, 1);
    grp = __shfl_sync(FULL, grp, 0);
    if (grp >= ngroups) break;
    const int w = grp * G + sub;
    const bool valid = w < d.W;
    const int wc = valid ? w : d.W - 1;
    const double* maos = d.minv_iso + (size_t)wc * (n + 1) * 2;      // [n+1][2], row n = 0 (ground / world anchor)
    const int nc = valid ? nj + d.c_count[wc] : 0;
    char* gs = reinterpret_cast<char*>(d.rec) + (size_t)grp * group_stride_bytes(d.nrec, G);
    const int R = d.grp_info[(size_t)grp * 4];                       // rounds of the group
    const unsigned bytes0 = (unsigned)d.grp_info[(size_t)grp * 4 + 1];   // bytes of round 0
    const unsigned stream_bytes = (unsigned)d.grp_info[(size_t)grp * 4 + 2];
    unsigned pf_pos = 0;                       // L2 prefetch cursor (bytes into the group stream)
    double* lam_out = d.lam_out + (size_t)wc * 3 * d.nrec;
    int* row_state = d.row_state + (size_t)wc * 3 * d.nrec;
    for (int i = sl; i < 6 * n; i += LPW) sb[i] = 0.0;

    bool active = nc > 0;
    double err = 0.0;
    int it = 0;
    unsigned probe_off = 0;                    // probe chunk: byte offset of its round in the group stream,
    int probe_meta = 0;                        //   first run | runs of the world << 6 | runs of the round << 12 | blocks of the round << 18
    double se = 0, s1 = 0, s2 = 0, s3 = 0;
    double best = -1.0;                        // exact pass: largest per-block contribution seen by this lane
    unsigned best_off = 0;
    int best_meta = 0;
    bool broken = false;                       // a header that is not a header: the group's solve stops, the worlds are flagged

    auto issue_round = [&](unsigned off, unsigned bytes) {          // one bulk copy feeds the whole warp-stage
      if (lane == 0) {
        mbar_arrive_tx(bar, bytes);
        bulk_g2s(stage_s, gs + off, bytes, bar, pol);
      }
    };

    if (R > 0 && bytes0 <= (unsigned)stage_cap && __any_sync(FULL, active)) {
      const double tol = d.prm.tol;
      const int k_max = d.prm.k_max;
      // One loop runs every phase (a single copy of the block code):
      //   PH_INIT   x0 = rhs scattered into the accumulator, round by round
      //   PH_PROBE  residual terms of one chunk per world: the cheap lower bound of the residual of x_k
      //   PH_EXACT  residual of x_k over all rounds (read-only; writes the lam_out / row_state taps)
      //   PH_UPDATE sweep k -> k+1, round by round
      // Round 0 is in flight when a round phase starts; nothing is in flight when it ends.
      int phase = PH_INIT, k = 0;
      bool need_exact = false;
      issue_round(0, bytes0);
      while (!broken) {
        const bool probe = (phase == PH_PROBE);
        const int mode = (phase == PH_INIT) ? MODE_INIT : (phase == PH_UPDATE ? MODE_UPDATE : MODE_RESID);
        const bool on = (phase == PH_EXACT) ? need_exact : active;
        const int nsteps = probe ? 1 : R;
        unsigned roff = 0;
        for (int t = 0; t < nsteps; t++) {
          // ---- the lane's run of this round into registers ----
          double2 rc[RCOLS];                   // run record
          double2 lm[RM][2];                   // multiplier sectors
          double2 bk[RM][BCOLS];               // block records
          int L = 0, jb[RM];
          unsigned cur_off;
          int cur_meta;
          if (probe) {
            // the world's probe chunk = the first blocks of the runs of one of its stages, read in place
            issue_round(0, bytes0);            // speculate "continue": round 0 streams in meanwhile
            const int ps = probe_meta & 63, pc = (probe_meta >> 6) & 63, pr = (probe_meta >> 12) & 63, pt = (probe_meta >> 18) & 255;
            cur_off = probe_off; cur_meta = probe_meta;
            const int j = ps + sl;
            jb[0] = j;
#pragma unroll
            for (int q = 1; q < RM; q++) jb[q] = 0;
            if (on && sl < pc) {
              L = 1;
              const char* lamp = gs + probe_off + HDRB;
              const char* runp = lamp + LAMB * pt;
              const char* blkp = runp + RUNB * pr;
              lm[0][0] = __ldcg(reinterpret_cast<const double2*>(lamp + LAMB * j));
              lm[0][1] = __ldcg(reinterpret_cast<const double2*>(lamp + LAMB * j) + 1);
#pragma unroll
              for (int c = 0; c < RCOLS; c++) rc[c] = __ldg(reinterpret_cast<const double2*>(runp + (c * pr + j) * 16));
#pragma unroll
              for (int c = 0; c < BCOLS; c++) bk[0][c] = __ldg(reinterpret_cast<const double2*>(blkp + (c * pt + j) * 16));
            }
          } else {
            mbar_wait(bar, parity);
            parity ^= 1u;
            const uint4 lens = *reinterpret_cast<const uint4*>(stage0);
            const uint4 meta = *reinterpret_cast<const uint4*>(stage0 + 16);
            const unsigned lw = (lane < 16) ? (lane < 8 ? lens.x : lens.y) : (lane < 24 ? lens.z : lens.w);
            L = (int)((lw >> ((lane & 7) * 4)) & 15u);
            unsigned m[RM];
            int total = 0, cnt0 = 0;
#pragma unroll
            for (int q = 0; q < RM; q++) {
              m[q] = __ballot_sync(FULL, L > q);
              jb[q] = total + __popc(m[q] & lt);
              if (q == 0) cnt0 = __popc(m[0]);
              total += __popc(m[q]);
            }
            const unsigned bytes = meta.x, nxt = meta.y;
            // range guard (the staged bytes become shared-memory and global addresses): the header must
            // describe exactly the bytes that were copied, and the next copy must fit the staging buffer
            if (__any_sync(FULL, L > RM) || bytes != runs_round_bytes(total, cnt0) || bytes > (unsigned)stage_cap || nxt > (unsigned)stage_cap) {
              if (sl == 0 && valid) atomicOr(&d.status[wc], 64);
              broken = true;
              break;
            }
            cur_off = roff;
            cur_meta = __popc(m[0] & ~wmask & lt) | (__popc(m[0] & wmask) << 6) | (cnt0 << 12) | (total << 18);
            if (phase == PH_INIT && t == 0) { probe_off = 0; probe_meta = cur_meta; }   // first probe: the world's stage 0
            if (!on) L = 0;
            if (L > 0) {
              const unsigned char* lamp = stage0 + HDRB;
              const unsigned char* runp = lamp + LAMB * total;
              const unsigned char* blkp = runp + RUNB * cnt0;
#pragma unroll
              for (int c = 0; c < RCOLS; c++) rc[c] = *reinterpret_cast<const double2*>(runp + (c * cnt0 + jb[0]) * 16);
#pragma unroll
              for (int q = 0; q < RM; q++) {
                if (L > q) {
                  lm[q][0] = *reinterpret_cast<const double2*>(lamp + LAMB * jb[q]);
                  lm[q][1] = *reinterpret_cast<const double2*>(lamp + LAMB * jb[q] + 16);
#pragma unroll
                  for (int c = 0; c < BCOLS; c++) bk[q][c] = *reinterpret_cast<const double2*>(blkp + (c * total + jb[q]) * 16);
                }
              }
            }
            // The staging buffer is handed back to the TMA unit here.  The loads above are generic-proxy
            // reads, the next copy is an async-proxy write: the two proxies are ordered only by a
            // cross-proxy fence (a generic fence is NOT enough, see egg_pgs_stream.cu / DESIGN.md).
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            __syncwarp();                          // staging buffer free again
            const unsigned roff_next = roff + bytes;
            if (t + 1 < R) issue_round(roff_next, nxt);
            if (pf > 0) {
              // HBM -> L2 prefetch cursor kept pf x 4 KB ahead of the consumer (one 128-byte line per
              // lane and span; the cursor wraps: the next sweep streams the same bytes again)
              int lead = (int)pf_pos - (int)roff_next;
              if (lead < 0) lead += (int)stream_bytes;
#pragma unroll
              for (int q = 0; q < 2; q++) {
                if (lead < pf * 4096) {
                  const unsigned a = pf_pos + lane * 128;
                  if (a < stream_bytes) prefetch_l2(gs + a);
                  pf_pos += 4096;
                  lead += 4096;
                  if (pf_pos >= stream_bytes) pf_pos = 0;
                }
              }
            }
            roff = roff_next;
          }

          // ---- the run: both bodies' accumulators stay in registers from its first block to its last ----
          if (L > 0) {
            const unsigned long long pkr = (unsigned long long)__double_as_longlong(rc[3].y);
            const int i0 = (int)(pkr & 1023u) - 1, i1 = (int)((pkr >> 10) & 1023u) - 1;
            if (i0 >= n || i1 >= n) { atomicOr(&d.status[wc], 64); L = 0; }   // a record that is not a record never becomes an address
            else {
              double Rc[9];
              egg_quat_rot(rc[0].x, rc[0].y, rc[1].x, rc[1].y, Rc);
              if ((pkr >> RK_JOINT) & 1u) {
#pragma unroll
                for (int q = 0; q < 9; q++) Rc[q] = -Rc[q];
              }
              const double dpx = rc[2].x, dpy = rc[2].y, dpz = rc[3].x;
              double2* q1 = reinterpret_cast<double2*>(sb + (i1 < 0 ? dummy : i1) * 6);
              double2* q0 = reinterpret_cast<double2*>(sb + (i0 < 0 ? dummy : i0) * 6);
              // accumulator pieces: (l.x,l.y) (l.z,a.x) (a.y,a.z); the ground / world side reads the all-zero dummy body
              double2 a1a = q1[0], a1b = q1[1], a1c = q1[2];
              double2 a0a = q0[0], a0b = q0[1], a0c = q0[2];
              double m1m, m1c, m0m, m0c;         // (1/m, 1/c) of the two bodies; the ground / anchor side is 0
              if (ISO == 2) {
                m1m = (i1 < 0) ? 0.0 : um; m1c = (i1 < 0) ? 0.0 : uc;
                m0m = (i0 < 0) ? 0.0 : um; m0c = (i0 < 0) ? 0.0 : uc;
              } else {
                const double2 t1 = ldg_keep(reinterpret_cast<const double2*>(maos + ((i1 < 0) ? n : i1) * 2), pol_keep);
                const double2 t0 = ldg_keep(reinterpret_cast<const double2*>(maos + ((i0 < 0) ? n : i0) * 2), pol_keep);
                m1m = t1.x; m1c = t1.y; m0m = t0.x; m0c = t0.y;
              }
#pragma unroll
              for (int q = 0; q < RM; q++) {
                if (L > q) {
                  const double x0 = lm[q][0].x, x1 = lm[q][0].y, x2 = lm[q][1].x;
                  const unsigned long long pkb = (unsigned long long)__double_as_longlong(lm[q][1].y);
                  const double r0x = bk[q][0].x, r0y = bk[q][0].y, r0z = bk[q][1].x;
                  const double ia0 = bk[q][1].y, ia1 = bk[q][2].x, ia2 = bk[q][2].y;
                  const double rh0 = bk[q][3].x, rh1 = bk[q][3].y, rh2 = bk[q][4].x;
                  const double r1x = r0x + dpx, r1y = r0y + dpy, r1z = r0z + dpz;
                  double d0, d1, d2;
                  if (mode == MODE_INIT) {
                    d0 = x0; d1 = x1; d2 = x2;
                  } else {
                    // t = J a = Rc ((l1 + a1 x r1) - (l0 + a0 x r0))
                    const double u1x = a1a.x + (a1c.x * r1z - a1c.y * r1y), u1y = a1a.y + (a1c.y * r1x - a1b.y * r1z), u1z = a1b.x + (a1b.y * r1y - a1c.x * r1x);
                    const double u0x = a0a.x + (a0c.x * r0z - a0c.y * r0y), u0y = a0a.y + (a0c.y * r0x - a0b.y * r0z), u0z = a0b.x + (a0b.y * r0y - a0c.x * r0x);
                    const double ux = u1x - u0x, uy = u1y - u0y, uz = u1z - u0z;
                    const double tx = Rc[0] * ux + Rc[1] * uy + Rc[2] * uz, ty = Rc[3] * ux + Rc[4] * uy + Rc[5] * uz, tz = Rc[6] * ux + Rc[7] * uy + Rc[8] * uz;
                    // e = rhs - (J a + cfm x) = -(A x - b) of the block's rows
                    const double e0 = (rh0 - cfm * x0) - tx, e1 = (rh1 - cfm * x1) - ty, e2 = (rh2 - cfm * x2) - tz;
                    if (mode == MODE_RESID) {
                      const int orig = (int)(pkb & 0xfffffu);
                      const bool eq = ((pkb >> BK_EQ) & 1u) != 0;
                      const double q0s = e0 * e0, q1s = e1 * e1, q2s = e2 * e2;
                      double c;
                      if (eq) { c = q0s + q1s + q2s; se += c; }
                      else {
                        // w = -e: at lo with w < 0, at hi with w > 0, strictly inside (sparse_iterations.cc:51-69)
                        const double c1 = ((x0 == -1.0 && e0 > 0) ? q0s : 0.0) + ((x1 == -1.0 && e1 > 0) ? q1s : 0.0) + ((x2 == 0.0 && e2 > 0) ? q2s : 0.0);
                        const double c2 = ((x0 == 1.0 && e0 < 0) ? q0s : 0.0) + ((x1 == 1.0 && e1 < 0) ? q1s : 0.0);
                        const double c3 = ((x0 > -1.0 && x0 < 1.0) ? q0s : 0.0) + ((x1 > -1.0 && x1 < 1.0) ? q1s : 0.0) + ((x2 > 0.0) ? q2s : 0.0);
                        s1 += c1; s2 += c2; s3 += c3;
                        c = c1 + c2 + c3;
                      }
                      if (q == 0 && c > best) { best = c; best_off = cur_off; best_meta = cur_meta; }   // the probe evaluates the first blocks of the runs
                      if (!probe) {                        // read-only pass over x_k: leave the taps in reference row order
                        if (orig < d.nrec) {
                          double* lo = lam_out + 3 * orig;
                          int* rs = row_state + 3 * orig;
                          lo[0] = x0; lo[1] = x1; lo[2] = x2;
                          rs[0] = eq ? 3 : (x0 == -1.0 ? 1 : (x0 == 1.0 ? 2 : 0));
                          rs[1] = eq ? 3 : (x1 == -1.0 ? 1 : (x1 == 1.0 ? 2 : 0));
                          rs[2] = eq ? 3 : (x2 == 0.0 ? 1 : 0);
                        }
                      }
                      continue;
                    }
                    // off-diagonal of the block's D (isotropic bodies): -(c0 q0 q0^T + c1 q1 q1^T), q = Rc r
                    const double g0x = Rc[0] * r0x + Rc[1] * r0y + Rc[2] * r0z, g0y = Rc[3] * r0x + Rc[4] * r0y + Rc[5] * r0z, g0z = Rc[6] * r0x + Rc[7] * r0y + Rc[8] * r0z;
                    const double g1x = Rc[0] * r1x + Rc[1] * r1y + Rc[2] * r1z, g1y = Rc[3] * r1x + Rc[4] * r1y + Rc[5] * r1z, g1z = Rc[6] * r1x + Rc[7] * r1y + Rc[8] * r1z;
                    const double h0x = m0c * g0x, h0y = m0c * g0y, h1x = m1c * g1x, h1y = m1c * g1y;
                    const double do0 = -(h0x * g0y + h1x * g1y);     // d10
                    const double do1 = -(h0x * g0z + h1x * g1z);     // d20
                    const double do2 = -(h0y * g0z + h1y * g1z);     // d21
                    // clamp kind of this block (q2 shift already folded in by the assembly kernel)
                    const bool contact = ((pkb >> BK_KIND) & 1u) == KIND_CONTACT;
                    const double lo01 = contact ? -1.0 : -kInf, hi01 = contact ? 1.0 : kInf, lo2 = contact ? 0.0 : -kInf;
                    double n0 = x0 + e0 * ia0;
                    n0 = clamp_sel(n0, lo01, hi01);
                    d0 = n0 - x0;
                    double n1 = x1 + (e1 - do0 * d0) * ia1;
                    n1 = clamp_sel(n1, lo01, hi01);
                    d1 = n1 - x1;
                    double n2 = x2 + ((e2 - do1 * d0) - do2 * d1) * ia2;
                    n2 = (n2 < lo2) ? lo2 : n2;
                    d2 = n2 - x2;
                    st_sector(reinterpret_cast<double*>(gs + cur_off + HDRB + (unsigned)(jb[q] * LAMB)), n0, n1, n2, lm[q][1].y);
                  }
                  // impulse scatter: a += M^-1 J^T delta
                  const double ix = Rc[0] * d0 + Rc[3] * d1 + Rc[6] * d2, iy = Rc[1] * d0 + Rc[4] * d1 + Rc[7] * d2, iz = Rc[2] * d0 + Rc[5] * d1 + Rc[8] * d2;
                  {
                    const double cx = r1y * iz - r1z * iy, cy = r1z * ix - r1x * iz, cz = r1x * iy - r1y * ix;   // r1 x imp
                    a1a.x += m1m * ix; a1a.y += m1m * iy; a1b.x += m1m * iz;
                    a1b.y += m1c * cx; a1c.x += m1c * cy; a1c.y += m1c * cz;
                  }
                  {
                    const double cx = r0y * iz - r0z * iy, cy = r0z * ix - r0x * iz, cz = r0x * iy - r0y * ix;   // r0 x imp
                    a0a.x -= m0m * ix; a0a.y -= m0m * iy; a0b.x -= m0m * iz;
                    a0b.y -= m0c * cx; a0c.x -= m0c * cy; a0c.y -= m0c * cz;
                  }
                }
              }
              if (mode != MODE_RESID) {
                if (i1 >= 0) { q1[0] = a1a; q1[1] = a1b; q1[2] = a1c; }
                if (i0 >= 0) { q0[0] = a0a; q0[1] = a0b; q0[2] = a0c; }
              }
            }
          }
          __syncwarp();                            // accumulator writes visible to the next round
        }
        if (broken) break;
        auto reduce4 = [&]() {
#pragma unroll
          for (int o = LPW / 2; o > 0; o >>= 1) {
            se += __shfl_xor_sync(FULL, se, o);
            s1 += __shfl_xor_sync(FULL, s1, o);
            s2 += __shfl_xor_sync(FULL, s2, o);
            s3 += __shfl_xor_sync(FULL, s3, o);
          }
        };
        if (probe) {
          reduce4();
          const double lb = sqrt(se) + (sqrt(s1) + sqrt(s2) + sqrt(s3));
          need_exact = active && !(lb > 2.0 * tol);
          se = s1 = s2 = s3 = 0.0;
          best = -1.0;
          if (!__any_sync(FULL, need_exact)) { phase = PH_UPDATE; if (active) ++it; }
          else phase = PH_EXACT;                   // rare; the round-0 copy in flight serves it as well
          continue;
        }
        // ---- phase transitions (warp-uniform) ----
        if (phase == PH_EXACT) {
          reduce4();
          if (need_exact) {
            err = sqrt(se) + (sqrt(s1) + sqrt(s2) + sqrt(s3));   // residual of x_k
            if (k >= k_max || !(err > tol)) active = false;      // x_k is final
          }
          // move the probe to the chunk with the largest contribution
          double bb = best;
          unsigned bo = best_off;
          int bc = best_meta;
#pragma unroll
          for (int o = LPW / 2; o > 0; o >>= 1) {
            const double ob = __shfl_xor_sync(FULL, bb, o);
            const unsigned oo = __shfl_xor_sync(FULL, bo, o);
            const int oc = __shfl_xor_sync(FULL, bc, o);
            if (ob > bb || (ob == bb && oo < bo)) { bb = ob; bo = oo; bc = oc; }
          }
          if (need_exact && bb > 0.0) { probe_off = bo; probe_meta = bc; }
          if (!__any_sync(FULL, active)) break;
          phase = PH_UPDATE;
          if (active) ++it;
          issue_round(0, bytes0);
          continue;
        }
        if (phase == PH_UPDATE) {
          // multipliers were written with generic stores; the async proxy reads them back next sweep
          asm volatile("fence.proxy.async.global;" ::: "memory");
          __syncwarp();
          ++k;
        }
        // after PH_INIT (k = 0) or PH_UPDATE: start the check of x_k
        se = s1 = s2 = s3 = 0.0;
        best = -1.0;
        if (k < k_max && __any_sync(FULL, active && ((probe_meta >> 6) & 63) > 0)) {
          phase = PH_PROBE;
        } else {
          phase = PH_EXACT;
          need_exact = active;
          issue_round(0, bytes0);
        }
      }
    } else if (R > 0 && bytes0 > (unsigned)stage_cap) {
      if (sl == 0 && valid) atomicOr(&d.status[wc], 64);
    }
    __syncwarp();

    if (valid) {
      if (sl == 0) {
        int* stt = d.stats + (size_t)w * 8;
        stt[4] = it;
        stt[5] = 0;
        stt[6] = (nc > 0 && cfm != 0.0);       // no rows: ComputeVDot is never reached (ensembles.cc:498-538)
        stt[7] = d.n_levels[w];
        d.resid[w] = err;
      }
      stream_integrate_world(d, w, sb, sl, LPW, dt);
    }
    __syncwarp();
  }
}

// Staging bytes for cap runs per world and stage: worst case every run is full.
size_t staging_bytes(int G, int cap) { return (size_t)HDRB + (size_t)G * cap * (RUNB + RUN_MAX * (LAMB + RBLKB)) + 32; }

template <int LPW, int ISO>
cudaError_t launch(const EggDev& d, double dt, cudaStream_t s) {
  constexpr int G = 32 / LPW;
  const size_t stg = staging_bytes(G, d.run_cap);
  const size_t smem = 64 + (size_t)G * 48 * d.n + stg;
  static thread_local size_t c_smem = ~(size_t)0;
  static thread_local int c_dev = -1, c_per_sm = 0, c_sms = 148;
  cudaError_t e = cudaSuccess;
  int dev = 0;
  EGG_FIRST(e, cudaGetDevice(&dev));
  if (e != cudaSuccess) return e;
  if (smem != c_smem || dev != c_dev) {
    EGG_FIRST(e, cudaFuncSetAttribute(egg_pgs_runs_kernel<LPW, ISO>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    EGG_FIRST(e, cudaDeviceGetAttribute(&c_sms, cudaDevAttrMultiProcessorCount, dev));
    EGG_FIRST(e, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&c_per_sm, egg_pgs_runs_kernel<LPW, ISO>, 32, smem));
    if (e != cudaSuccess) return e;
    if (c_per_sm < 1) return cudaErrorLaunchOutOfResources;
    c_smem = smem; c_dev = dev;
  }
  int per_sm = c_per_sm;
  if (d.sel.ctas_per_sm > 0 && d.sel.ctas_per_sm < per_sm) per_sm = d.sel.ctas_per_sm;
  const int groups = (d.W + G - 1) / G;
  const int grid = groups < c_sms * per_sm ? groups : c_sms * per_sm;
  e = cudaMemsetAsync(d.work_ctr, 0, sizeof(int), s);
  if (e != cudaSuccess) return e;
  egg_pgs_runs_kernel<LPW, ISO><<<grid, 32, smem, s>>>(d, dt, d.sel.pf, (int)(stg - 32));
  return cudaGetLastError();
}

template <int ISO>
cudaError_t launch_lpw(const EggDev& d, double dt, cudaStream_t s) {
  switch (d.lpw) {
    case 1: return launch<1, ISO>(d, dt, s);
    case 2: return launch<2, ISO>(d, dt, s);
    case 4: return launch<4, ISO>(d, dt, s);
    default: return launch<8, ISO>(d, dt, s);
  }
}

}  // namespace

// The run format applies to FP64 records of isotropic bodies with at most 8 lanes per world.
int egg_runs_rmax(const EggDev& d) {
  // EGG_PGS_RUNS (d.sel.runs) is a development override of EGG_OPT_PGS_RUNS (quirks bit 16)
  const bool want = d.sel.runs >= 0 ? d.sel.runs != 0 : (d.prm.quirks & 16) != 0;
  if (!want || !d.rec_fmt || !d.st_runs || d.iso < 1 || d.lpw > 8 || d.blkb != RECB64 + LAMB) return 0;
  return RUN_MAX;
}

// Runs per world and stage: the lanes of the world, unless the staging buffer they need would cost
// resident warps (64-body worlds: 11 one-warp CTAs per SM with 4 x 64 x 48 B of accumulators each
// leave ~7.7 KB for the staging buffer: 6 runs per world and stage instead of 8).
int egg_run_cap(const EggDev& d) {
  const int G = 32 / d.lpw;
  if (d.sel.run_cap > 0) return d.sel.run_cap < d.lpw ? d.sel.run_cap : d.lpw;
  const long long per_cta = 232448 / d.sel.target_ctas - 1024;
  const long long avail = per_cta - 64 - (long long)G * 48 * d.n - HDRB - 32;
  int cap = (int)(avail / ((long long)G * (RUNB + RUN_MAX * (LAMB + RBLKB))));
  if (cap > d.lpw) cap = d.lpw;
  const int floor_cap = d.lpw > 1 ? d.lpw / 2 : 1;
  if (cap < floor_cap) cap = floor_cap;
  return cap;
}

size_t egg_runs_smem(const EggDev& d) { return 64 + (size_t)(32 / d.lpw) * 48 * d.n + staging_bytes(32 / d.lpw, d.lpw); }

// Rounds + records of the run format (the schedule kernel of egg_pgs_stream.cu has run before).
cudaError_t egg_launch_assemble_runs_tail(const EggDev& d, double dt, cudaStream_t s) {
  const int G = 32 / d.lpw;
  cudaError_t e = cudaSuccess;
  const int ngroups = (d.W + G - 1) / G;
  egg_rounds_runs_kernel<<<(ngroups + 3) / 4, 128, 0, s>>>(d, G);
  const size_t smem = (size_t)(EGG_DYN + EGG_STAT + 6) * d.n * sizeof(double);
  const int nt = egg_records_threads(d);    // 32, 128 or 256, by the rule of the group stream (egg_pgs_stream.cu)
  if (nt == 32) {
    if (smem > 48 * 1024) EGG_FIRST(e, cudaFuncSetAttribute(egg_records_runs_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    if (e != cudaSuccess) return e;
    egg_records_runs_kernel<32><<<d.W, 32, smem, s>>>(d, dt, G);
  } else if (nt == 128) {
    if (smem > 48 * 1024) EGG_FIRST(e, cudaFuncSetAttribute(egg_records_runs_kernel<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    if (e != cudaSuccess) return e;
    egg_records_runs_kernel<128><<<d.W, 128, smem, s>>>(d, dt, G);
  } else {
    if (smem > 48 * 1024) EGG_FIRST(e, cudaFuncSetAttribute(egg_records_runs_kernel<256>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    if (e != cudaSuccess) return e;
    egg_records_runs_kernel<256><<<d.W, 256, smem, s>>>(d, dt, G);
  }
  return cudaGetLastError();
}

cudaError_t egg_launch_solve_pgs_runs(const EggDev& d, double dt, cudaStream_t s) {
  if (d.iso == 2) return launch_lpw<2>(d, dt, s);
  return launch_lpw<1>(d, dt, s);
}
