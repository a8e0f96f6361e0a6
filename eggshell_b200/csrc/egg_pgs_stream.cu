// Variant "stream" of the projected Gauss-Seidel solve (default) and its group-stream assembly.
//
// What the profiles said, step by step (profiles/r1d..r1f, DESIGN.md section 4):
//   * "fast" variant: latency-bound, worlds in flight per SM capped by shared memory (112 B per
//     body: accumulator + the frozen copy the fused residual needs) and 227 registers.
//   * first "stream" version (48 B per body, 11 resident warps): 1.8x faster, but throughput no
//     longer moved with occupancy (6..11 warps/SM: same time) nor with the M^-1 variant: the record
//     stream was bound by DRAM *efficiency*.  tools/micro/dram_chunk_bench: random contiguous reads
//     of 960 B reach 3.4 TB/s on this part, 3840 B 5.4 TB/s, 7680 B 7.0 TB/s; a stage of one
//     world is ~1 KB.
// Hence this layout: the G = 32/LPW worlds that share a warp are interleaved in memory round by
// round ("group stream"), so that ONE bulk copy of ~4 KB feeds a whole warp-stage.
//
//   group stream = for round t = 0..R-1:
//       [64-byte header][32-byte multiplier sector of every block of the round][records of world 0's
//       stage t]...[records of world G-1's stage t]            (padded to a multiple of 32 B)
//   header: u8 start[s] (block index of world s inside the round, start[G] = total), bytes 40 / 41 =
//   totals of the next two rounds (cyclic), so the size of the next copy is known one round ahead.
//
// Algorithm (unchanged in exact arithmetic, reference row order inside every world):
//   * No frozen accumulator.  The reference evaluates the residual of x_k after every sweep only to
//     decide "stop / continue" (sparse_iterations.cc:196-215).  The residual is a sum of norms of
//     non-negative per-row terms (sparse_iterations.cc:51-69), so the same formula over ANY subset
//     of blocks is a lower bound.  Before each sweep one chunk of <= LPW blocks per world (the
//     "probe") is evaluated against a = a_k (nothing has been updated yet, so no copy is needed);
//     if that partial residual already exceeds 2 tol the decision "continue" is certain and the
//     sweep runs without any residual work.  Otherwise the full residual is evaluated exactly
//     (one read-only pass) and the reference's decision is taken on it; the probe then moves to
//     the chunk that contributed most.  Sweep counts, final multipliers and the reported
//     residual are those of the reference algorithm.
//   * The row update is written in increment form  x' = x + (rhs - J a - cfm x) / (D + cfm),  so
//     only 1/(D+cfm) is stored.  The multipliers are staged with their round (one 32-byte sector
//     per block, contiguous per round) and written back in place with full-sector stores; the
//     read-only pass that ends a world's solve also writes them out in reference row order
//     (lam_out / row_state taps).
//   * Ordering between this warp's shared-memory loads of a stage and the TMA copy of the next
//     one is a cross-proxy fence (fence.proxy.async.shared::cta), see the comment at the fence.
//   * World groups are handed out by an atomic counter.
//
// Per warp: 64 B + G x n x 48 B accumulators + 64 B + G x LPW x 208 B staging.  64-body worlds:
// 19072 B -> 11 resident warps of 4 worlds per SM at 164 registers.
//
// Replaces: sparse::GaussSeidelIteration + GetResidualError + the velocity/position update, i.e.
// /root/reference/eggshell/sparse_iterations.cc:148-226,51-69,
// sparse_iterations_utils.cc:12-21,159-243,495-695, ensembles.cc:535,572-591; the assembly kernels
// replace Ensemble::ComputeJ / rhs (ensembles.cc:38-87,156-171,563-570) via egg_record.cuh.
#include "egg_internal.cuh"
#include "egg_record.cuh"
#include "egg_stream.cuh"
#include <cstdlib>

namespace {

// ---------------------------------------------------------------------------------------------
// Assembly 1/3: dependency levels and stages of one world (one warp per world, lane 0 scans).
//   level(c) = 1 + max level of earlier constraints sharing a body  (constraints in reference
//   order: joints, then contacts, ensembles.cc:234-239); a level is cut into stages of <= cap.
// rm > 0 (egg_pgs_runs.cu): the unit is a RUN of up to rm consecutive constraints on the same
//   ordered body pair (the contacts of one manifold, ensembles.cc:449-473): they would occupy
//   consecutive levels anyway, and one lane can carry both bodies' accumulators through them.
// Out: c_pos[c] = stage << 8 | lane << 3 | index inside the run, st_cnt[stage] (rm == 1) or
//   st_runs[stage] (4 bits per lane: run length), n_levels = #stages.
__global__ void __launch_bounds__(128) egg_schedule_kernel(EggDev d, int cap, int wpc, int rm) {
  extern __shared__ __align__(16) unsigned char sm_raw[];
  const int wl = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int w = blockIdx.x * wpc + wl;
  const int n = d.n, nj = d.nj, nrec = d.nrec;
  // per world: blast[n] | lev[nrec] | pos[nrec] | lcnt[nrec+1] | lstage[nrec+1]   (all u16)
  const size_t per = (size_t)(n + 4 * nrec + 2 + 7) & ~(size_t)7;
  unsigned short* blast = reinterpret_cast<unsigned short*>(sm_raw) + (size_t)wl * per;
  unsigned short* lev = blast + n;
  unsigned short* pos = lev + nrec;     // unit index inside its level (bits 0..11 when rm > 0: | k << 12 | last-of-run << 15)
  unsigned short* lcnt = pos + nrec;
  unsigned short* lstage = lcnt + nrec + 1;
  if (wl >= wpc || w >= d.W) return;
  const int nc = nj + d.c_count[w];
  const int* c_i0 = d.c_i0 + (size_t)w * d.maxc;
  const int* c_i1 = d.c_i1 + (size_t)w * d.maxc;
  for (int b = lane; b < n; b += 32) blast[b] = 0;          // level + 1 of the last unit on the body (0 = none)
  for (int c = lane; c <= nc; c += 32) lcnt[c] = 0;
  // body indices + 1 of every constraint, staged with coalesced loads: the serial scan below must not
  // wait for global memory once per constraint (lev[c] is overwritten by the scan, lstage after it)
  for (int c = lane; c < nc; c += 32) {
    int i0, i1;
    if (c < nj) { i0 = d.j_i0[(size_t)w * nj + c]; i1 = d.j_i1[(size_t)w * nj + c]; }
    else { i0 = __ldg(c_i0 + c - nj); i1 = __ldg(c_i1 + c - nj); }
    lev[c] = (unsigned short)(i0 + 1);
    lstage[c] = (unsigned short)(i1 + 1);
  }
  if (rm > 0) {
    // pos[c] = 1: contact c may extend the run of contact c - 1: same ordered body pair and bit-identical
    // normal (one manifold, or one body's ground contacts), so the two share the contact frame
    const double* gm = d.c_geom + (size_t)w * 7 * d.maxc;
    for (int c = lane; c < nc; c += 32) {
      bool same = false;
      if (c > nj) {
        const int k = c - nj;
        same = c_i0[k] == c_i0[k - 1] && c_i1[k] == c_i1[k - 1];
        for (int q = 3; q < 6 && same; q++) same = __double_as_longlong(gm[(size_t)q * d.maxc + k]) == __double_as_longlong(gm[(size_t)q * d.maxc + k - 1]);
      }
      pos[c] = same ? 1 : 0;
    }
  }
  __syncwarp();
  int nl = 0, ns = 0;
  if (lane == 0) {
    int pl = 0, pp = 0, plen = 0;
    for (int c = 0; c < nc; c++) {
      const int i0 = (int)lev[c] - 1, i1 = (int)lstage[c] - 1;
      if (rm > 0 && pos[c] != 0 && plen < rm) {                         // extends the previous run
        pos[c - 1] &= 0x7fff;                                            // the previous block is no longer the last
        lev[c] = (unsigned short)pl;
        pos[c] = (unsigned short)(pp | (plen << 12) | 0x8000);
        plen++;
        continue;
      }
      int l = 0;
      if (i0 >= 0) l = blast[i0];
      if (i1 >= 0) l = max(l, (int)blast[i1]);
      if (i0 >= 0) blast[i0] = (unsigned short)(l + 1);
      if (i1 >= 0) blast[i1] = (unsigned short)(l + 1);
      lev[c] = (unsigned short)l;
      pp = lcnt[l]++;
      pos[c] = (unsigned short)((rm > 0) ? (pp | 0x8000) : pp);
      pl = l; plen = 1;
      nl = max(nl, l + 1);
    }
    unsigned char* sc = d.st_cnt + (size_t)w * nrec;
    for (int l = 0; l < nl; l++) {
      const int cnt = lcnt[l];
      lstage[l] = (unsigned short)ns;
      for (int k = 0; k < cnt; k += cap) sc[ns++] = (unsigned char)min(cap, cnt - k);
    }
    d.n_levels[w] = ns;
  }
  ns = __shfl_sync(0xffffffffu, ns, 0);
  __syncwarp();
  int* cp = d.c_pos + (size_t)w * nrec;
  if (rm > 0) {
    unsigned* sr = d.st_runs + (size_t)w * nrec;
    for (int t = lane; t < ns; t += 32) sr[t] = 0u;
    __syncwarp();
    for (int c = lane; c < nc; c += 32) {
      const int pv = pos[c], p = pv & 0xfff, k = (pv >> 12) & 7;
      const int stg = lstage[lev[c]] + p / cap, ln = p % cap;
      cp[c] = (stg << 8) | (ln << 3) | k;
      if (pv & 0x8000) atomicOr(sr + stg, (unsigned)(k + 1) << (4 * ln));   // the last block of a run knows its length
    }
  } else {
    for (int c = lane; c < nc; c += 32) {
      const int p = pos[c];
      cp[c] = ((lstage[lev[c]] + p / cap) << 8) | ((p % cap) << 3);
    }
  }
}

// Assembly 2/3: round offsets and headers of one group (one warp per group).
__global__ void __launch_bounds__(128) egg_rounds_kernel(EggDev d, int G) {
  const int g = blockIdx.x * 4 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  const int ngroups = (d.W + G - 1) / G;
  if (g >= ngroups) return;
  const int nrec = d.nrec;
  int R = 0;
  for (int s = 0; s < G; s++) { const int w = g * G + s; if (w < d.W) R = max(R, d.n_levels[w]); }
  unsigned char* gs = reinterpret_cast<unsigned char*>(d.rec) + (size_t)g * group_stride_bytes(nrec, G);
  unsigned* roff = d.round_off + (size_t)g * (nrec + 1);
  auto total_of = [&](int t) -> int {
    int tot = 0;
    for (int s = 0; s < G; s++) { const int w = g * G + s; if (w < d.W && t < d.n_levels[w]) tot += d.st_cnt[(size_t)w * nrec + t]; }
    return tot;
  };
  unsigned base = 0;
  for (int t0 = 0; t0 < R; t0 += 32) {
    const int t = t0 + lane;
    unsigned char hdr[HDRB];
#pragma unroll
    for (int k = 0; k < HDRB; k++) hdr[k] = 0;
    int tot = 0;
    if (t < R) {
      for (int s = 0; s < G; s++) {
        const int w = g * G + s;
        hdr[s] = (unsigned char)tot;
        if (w < d.W && t < d.n_levels[w]) tot += d.st_cnt[(size_t)w * nrec + t];
      }
      hdr[G] = (unsigned char)tot;
      hdr[HDR_NEXT] = (unsigned char)total_of((t + 1) % R);
      hdr[HDR_NEXT + 1] = (unsigned char)total_of((t + 2) % R);
    }
    const unsigned bytes = (t < R) ? round_bytes(tot, d.blkb) : 0u;
    unsigned incl = bytes;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const unsigned v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += v; }
    const unsigned off = base + incl - bytes;
    if (t < R) {
      roff[t] = off;
      uint4* hp = reinterpret_cast<uint4*>(gs + off);
      const uint4* hs = reinterpret_cast<const uint4*>(hdr);
#pragma unroll
      for (int q = 0; q < HDRB / 16; q++) hp[q] = hs[q];
    }
    base += __shfl_sync(0xffffffffu, incl, 31);
  }
  if (lane == 0) {
    int* gi = d.grp_info + (size_t)g * 4;
    gi[0] = R;
    gi[1] = (R > 0) ? total_of(0) : 0;
    gi[2] = (int)base;
    gi[3] = (R > 0) ? total_of(1 % R) : 0;
  }
}

// Assembly 3/3: one CTA per world builds the records and writes them at their round positions.
template <int NT>
__global__ void __launch_bounds__(NT, (NT >= 256) ? 2 : 4) egg_records_kernel(EggDev d, double dt, int G) {
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
  const int g = w / G, sub = w % G;
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
    const int p = cp[c], stg = p >> 8, idx = (p >> 3) & 31;
    const unsigned ro = roff[stg];
    const unsigned start = gs[ro + sub];
    const int kind = __double2hiint(v[REC_META]);
    const unsigned long long pk = (unsigned long long)(i0 + 1) | ((unsigned long long)(i1 + 1) << 10) | ((unsigned long long)kind << 20) | ((unsigned long long)c << 21);
    const unsigned total = gs[ro + G];
    double2* lam = reinterpret_cast<double2*>(gs + ro + HDRB + (size_t)LAMB * (start + idx));
    lam[0] = make_double2(v[REC_RHS], v[REC_RHS + 1]);              // x0 = rhs
    lam[1] = make_double2(v[REC_RHS + 2], __longlong_as_double((long long)pk));
    const int recb = d.blkb - LAMB;
    unsigned char* rp = gs + ro + HDRB + (size_t)LAMB * total + (size_t)recb * (start + idx);
    if (recb == RECB64) {
      double o[SREC];
#pragma unroll
      for (int q = 0; q < 6; q++) o[q] = v[q];                      // rows 0 and 1 of Rc (row 2 = +-(row 0 x row 1))
#pragma unroll
      for (int q = 0; q < 9; q++) o[6 + q] = v[9 + q];              // r0, r1, D off-diagonal
#pragma unroll
      for (int q = 0; q < 3; q++) { o[15 + q] = v[REC_INVA + q]; o[18 + q] = v[REC_RHS + q]; }
      o[21] = 0.0;
      double2* out = reinterpret_cast<double2*>(rp);
#pragma unroll
      for (int q = 0; q < SREC / 2; q++) out[q] = make_double2(o[2 * q], o[2 * q + 1]);
    } else {
      // precision = 32: the constraint data in FP32 (multipliers, accumulators and arithmetic stay FP64)
      float o[24];
#pragma unroll
      for (int q = 0; q < 18; q++) o[q] = (float)v[q];
#pragma unroll
      for (int q = 0; q < 3; q++) { o[18 + q] = (float)v[REC_INVA + q]; o[21 + q] = (float)v[REC_RHS + q]; }
      float4* out = reinterpret_cast<float4*>(rp);
#pragma unroll
      for (int q = 0; q < 6; q++) out[q] = make_float4(o[4 * q], o[4 * q + 1], o[4 * q + 2], o[4 * q + 3]);
      reinterpret_cast<double2*>(rp)[6] = make_double2(__longlong_as_double((long long)pk), 0.0);
    }
  }
}

enum { MODE_INIT = 0, MODE_UPDATE = 1, MODE_RESID = 2 };
enum { PH_INIT = 0, PH_PROBE = 1, PH_EXACT = 2, PH_UPDATE = 3 };

// ISO >= 1: every body's M^-1 is (1/m) I3, (1/c) I3 exactly (egg_init snaps numerically isotropic
// inverse inertias, see egg_solve.cu) and comes as one 16-byte load per body.  ISO == 2: all
// bodies of the batch share the same (1/m, 1/c) (every body of the reference is the same cube,
// body.h:91) and the pair is a kernel constant.
//
// COULOMB (egg_set_friction): the tangent rows of a block projected as a contact are bounded by
// [-b, b], b = mu[w] max(x_n, 0), x_n = the block's normal multiplier before its update (x2), instead
// of [-1, 1].  Such a bound moves with the normal, so "x equals its bound" is recorded by each update
// as a clamp flag per tangent row (0 free, 1 at -b, 2 at +b) in bits PK_FLAGS.. of the packed word of
// the multiplier sector; the residual and the row_state taps read the flags.  Every decode of the
// packed word reads (int)(pk >> 21), i.e. bits 21..52, so the flags never reach an index.
constexpr int PK_FLAGS = 56;
template <int LPW, int MINB, int ISO, bool F32, bool COULOMB>
__global__ void __launch_bounds__(32, MINB) egg_pgs_stream_kernel(EggDev d, double dt, int pf, const double* __restrict__ mu_w) {
  constexpr int G = 32 / LPW;
  constexpr int RECB = F32 ? RECB32 : RECB64;   // bytes of one staged record
  constexpr int SPIECES = RECB / 16;
  constexpr int BLKB = RECB + LAMB;
  extern __shared__ __align__(128) unsigned char smraw[];
  const int n = d.n, lane = threadIdx.x, sub = lane / LPW, sl = lane % LPW;
  // shared memory: [mbarrier probes 8 B][mbarrier rounds, buffer 0, 8 B][dummy body 48 B: the ground / world
  //                anchor, always zero][G x n x 6 doubles accumulators][64 B header + G x LPW x (32 + 176) B staging]
  const unsigned bar2 = s32(smraw), bar = s32(smraw + 8);
  double* sb = reinterpret_cast<double*>(smraw + 64) + (size_t)sub * 6 * n;
  const int dummy = -(sub * n) - 1;            // body index of the dummy relative to this world's sb
  unsigned char* stage0 = smraw + 64 + (size_t)G * 48 * n;
  const unsigned stage_s = s32(stage0);
  const double cfm = d.prm.cfm;
  const int nj = d.nj;
  const unsigned FULL = 0xffffffffu;

  if (lane == 0) {
    mbar_init(bar, 1);
    mbar_init(bar2, G);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (lane < 6) reinterpret_cast<double*>(smraw + 16)[lane] = 0.0;
  const unsigned long long pol = policy_evict_first();
  const unsigned long long pol_keep = policy_evict_last();
  double um = 0.0, uc = 0.0;                   // ISO == 2: the batch-wide (1/m, 1/c)
  if (ISO == 2) { um = d.minv_iso[0]; uc = d.minv_iso[1]; }
  __syncwarp();
  unsigned parity = 0, parity2 = 0;
  const int ngroups = (d.W + G - 1) / G;

  while (true) {
    int grp = 0;
    if (lane == 0) grp = atomicAdd(d.work_ctr, 1);
    grp = __shfl_sync(FULL, grp, 0);
    if (grp >= ngroups) break;
    const int w = grp * G + sub;
    const bool valid = w < d.W;
    const int wc = valid ? w : d.W - 1;
    const double* maos = ISO ? d.minv_iso + (size_t)wc * (n + 1) * 2      // [n+1][2], row n = 0 (ground / world anchor)
                             : d.minv_aos + (size_t)wc * (n + 1) * 10;    // [n+1][10]
    const int nc = valid ? nj + d.c_count[wc] : 0;
    const double mu = COULOMB ? mu_w[wc] : 0.0;
    char* gs = reinterpret_cast<char*>(d.rec) + (size_t)grp * group_stride_bytes(d.nrec, G);
    const int R = d.grp_info[(size_t)grp * 4];                // rounds of the group
    const int tot0 = d.grp_info[(size_t)grp * 4 + 1];         // blocks in round 0
    const unsigned stream_bytes = (unsigned)d.grp_info[(size_t)grp * 4 + 2];
    unsigned pf_pos = 0;                       // L2 prefetch cursor (bytes into the group stream)
    double* lam_out = d.lam_out + (size_t)wc * 3 * d.nrec;
    int* row_state = d.row_state + (size_t)wc * 3 * d.nrec;
    for (int i = sl; i < 6 * n; i += LPW) sb[i] = 0.0;

    bool active = nc > 0;
    double err = 0.0;
    int it = 0;
    unsigned probe_off = 0;                    // probe chunk: byte offset of its round in the group stream,
    int probe_meta = 0;                        //   start | total << 8 | count << 16 of the world's blocks in that round
    int probe_cnt = 0;
    double se = 0, s1 = 0, s2 = 0, s3 = 0;
    double best = -1.0;                        // exact pass: largest per-block contribution seen by this lane
    unsigned best_off = 0;
    int best_meta = 0;

    auto issue_round = [&](unsigned off, int total) {          // one bulk copy feeds the whole warp-stage
      if (lane == 0) {
        const unsigned bytes = round_bytes(total, BLKB);
        mbar_arrive_tx(bar, bytes);
        bulk_g2s(stage_s, gs + off, bytes, bar, pol);
      }
    };
    auto start_rounds = [&]() { issue_round(0, tot0); };      // round 0 of a pass
    auto issue_probe = [&](bool on) {                       // every world leader arrives exactly once
      if (sl == 0) {
        if (on && probe_cnt > 0) {
          // the world's multipliers and records of the probe round, into its own slices of the staging buffer
          const int ps = probe_meta & 255, pt = (probe_meta >> 8) & 255;
          mbar_arrive_tx(bar2, (unsigned)(BLKB * probe_cnt));
          bulk_g2s(stage_s + HDRB + sub * (LPW * LAMB), gs + probe_off + HDRB + ps * LAMB, (unsigned)(LAMB * probe_cnt), bar2, pol);
          bulk_g2s(stage_s + HDRB + 32 * LAMB + sub * (LPW * RECB), gs + probe_off + HDRB + pt * LAMB + ps * RECB, (unsigned)(RECB * probe_cnt), bar2, pol);
        } else {
          mbar_arrive(bar2);
        }
      }
    };

    // One block on record v.  MODE_INIT: a = M^-1 J^T x0 (x0 = rhs, already in the record);
    // MODE_UPDATE: projected row-by-row update + impulse scatter; MODE_RESID: residual terms only.
    auto step = [&](const double2* v, double x0, double x1, double x2, unsigned long long pk_lam, int mode, bool mine, unsigned lam_off, unsigned round_off, int round_meta, bool finalize) {
      if (!mine) return;
      double fld[24];
      unsigned long long pk;
      if (F32) {
#pragma unroll
        for (int q = 0; q < 6; q++) {
          const float2 lo = *reinterpret_cast<const float2*>(&v[q].x), hi = *reinterpret_cast<const float2*>(&v[q].y);
          fld[4 * q] = (double)lo.x; fld[4 * q + 1] = (double)lo.y; fld[4 * q + 2] = (double)hi.x; fld[4 * q + 3] = (double)hi.y;
        }
        pk = (unsigned long long)__double_as_longlong(v[6].x);
      } else {
#pragma unroll
        for (int q = 0; q < 3; q++) { fld[2 * q] = v[q].x; fld[2 * q + 1] = v[q].y; }                  // Rc rows 0, 1
#pragma unroll
        for (int q = 3; q < 11; q++) { fld[3 + 2 * q] = v[q].x; if (q < 10) fld[4 + 2 * q] = v[q].y; }   // r0 .. rhs -> fld[9..23]
        pk = pk_lam;
        // row 2 of the frame: a rotation's third row is row 0 x row 1; a joint's frame is -I (det -1)
        const double sg = ((int)(pk >> 21) < nj) ? -1.0 : 1.0;
        fld[6] = sg * (fld[1] * fld[5] - fld[2] * fld[4]);
        fld[7] = sg * (fld[2] * fld[3] - fld[0] * fld[5]);
        fld[8] = sg * (fld[0] * fld[4] - fld[1] * fld[3]);
      }
      const int i0 = (int)(pk & 1023u) - 1, i1 = (int)((pk >> 10) & 1023u) - 1;
      // range guard: a record that is not a record must never become an address (three compares per
      // block; the world is flagged EGG_ST_INTERNAL instead)
      if (i0 >= n || i1 >= n || (int)(pk >> 21) >= d.nrec) { atomicOr(&d.status[wc], 64); return; }
      const int j0 = (i0 < 0) ? n : i0, j1 = (i1 < 0) ? n : i1;
      // accumulator pieces: (l.x,l.y) (l.z,a.x) (a.y,a.z); the ground / world side reads the
      // all-zero dummy body (never written: its stores are predicated off below)
      double2* q1 = reinterpret_cast<double2*>(sb + (i1 < 0 ? dummy : i1) * 6);
      double2* q0 = reinterpret_cast<double2*>(sb + (i0 < 0 ? dummy : i0) * 6);
      double2 a1a = q1[0], a1b = q1[1], a1c = q1[2];
      double2 a0a = q0[0], a0b = q0[1], a0c = q0[2];
      constexpr int MN = ISO ? 2 : 10;
      double m1[MN], m0[MN];
      if (ISO == 2) {
        m1[0] = m0[0] = um; m1[1] = m0[1] = uc;
      } else if (mode != MODE_RESID) {          // M^-1 of both bodies: issued early, used in the scatter
        const double2* mq1 = reinterpret_cast<const double2*>(maos + j1 * MN);
        const double2* mq0 = reinterpret_cast<const double2*>(maos + j0 * MN);
#pragma unroll
        for (int p = 0; p < MN / 2; p++) {
          const double2 t1 = ldg_keep(mq1 + p, pol_keep), t0 = ldg_keep(mq0 + p, pol_keep);
          m1[2 * p] = t1.x; m1[2 * p + 1] = t1.y; m0[2 * p] = t0.x; m0[2 * p + 1] = t0.y;
        }
      }
      double d0, d1, d2;
      if (mode == MODE_INIT) {
        d0 = x0; d1 = x1; d2 = x2;
      } else {
        // t = J a = Rc ((l1 + a1 x r1) - (l0 + a0 x r0))
        const double u1x = a1a.x + (a1c.x * R1Z - a1c.y * R1Y), u1y = a1a.y + (a1c.y * R1X - a1b.y * R1Z), u1z = a1b.x + (a1b.y * R1Y - a1c.x * R1X);
        const double u0x = a0a.x + (a0c.x * R0Z - a0c.y * R0Y), u0y = a0a.y + (a0c.y * R0X - a0b.y * R0Z), u0z = a0b.x + (a0b.y * R0Y - a0c.x * R0X);
        const double ux = u1x - u0x, uy = u1y - u0y, uz = u1z - u0z;
        const double tx = RC0 * ux + RC1 * uy + RC2 * uz, ty = RC3 * ux + RC4 * uy + RC5 * uz, tz = RC6 * ux + RC7 * uy + RC8 * uz;
        // e = rhs - (J a + cfm x) = -(A x - b) of the block's rows
        const double e0 = (RH0 - cfm * x0) - tx, e1 = (RH1 - cfm * x1) - ty, e2 = (RH2 - cfm * x2) - tz;
        if (mode == MODE_RESID) {
          const int orig = (int)(pk >> 21);
          const bool eq = orig < nj;
          const double q0s = e0 * e0, q1s = e1 * e1, q2s = e2 * e2;
          double c;
          if (eq) { c = q0s + q1s + q2s; se += c; }
          else if (COULOMB) {
            // the tangent rows by the clamp flags of the update that produced x_k (none for x_0: free)
            const unsigned f0 = (unsigned)(pk_lam >> PK_FLAGS) & 3u, f1 = (unsigned)(pk_lam >> (PK_FLAGS + 2)) & 3u;
            const double c1 = ((f0 == 1u && e0 > 0) ? q0s : 0.0) + ((f1 == 1u && e1 > 0) ? q1s : 0.0) + ((x2 == 0.0 && e2 > 0) ? q2s : 0.0);
            const double c2 = ((f0 == 2u && e0 < 0) ? q0s : 0.0) + ((f1 == 2u && e1 < 0) ? q1s : 0.0);
            const double c3 = ((f0 == 0u) ? q0s : 0.0) + ((f1 == 0u) ? q1s : 0.0) + ((x2 > 0.0) ? q2s : 0.0);
            s1 += c1; s2 += c2; s3 += c3;
            c = c1 + c2 + c3;
          } else {
            // w = -e: at lo with w < 0, at hi with w > 0, strictly inside (sparse_iterations.cc:51-69)
            const double c1 = ((x0 == -1.0 && e0 > 0) ? q0s : 0.0) + ((x1 == -1.0 && e1 > 0) ? q1s : 0.0) + ((x2 == 0.0 && e2 > 0) ? q2s : 0.0);
            const double c2 = ((x0 == 1.0 && e0 < 0) ? q0s : 0.0) + ((x1 == 1.0 && e1 < 0) ? q1s : 0.0);
            const double c3 = ((x0 > -1.0 && x0 < 1.0) ? q0s : 0.0) + ((x1 > -1.0 && x1 < 1.0) ? q1s : 0.0) + ((x2 > 0.0) ? q2s : 0.0);
            s1 += c1; s2 += c2; s3 += c3;
            c = c1 + c2 + c3;
          }
          if (c > best) { best = c; best_off = round_off; best_meta = round_meta; }
          if (finalize) {                          // read-only pass over x_k: leave the taps in reference row order
            double* lo = lam_out + 3 * orig;
            int* rs = row_state + 3 * orig;
            lo[0] = x0; lo[1] = x1; lo[2] = x2;
            if (COULOMB) {
              rs[0] = eq ? 3 : (int)((pk_lam >> PK_FLAGS) & 3u);
              rs[1] = eq ? 3 : (int)((pk_lam >> (PK_FLAGS + 2)) & 3u);
            } else {
              rs[0] = eq ? 3 : (x0 == -1.0 ? 1 : (x0 == 1.0 ? 2 : 0));
              rs[1] = eq ? 3 : (x1 == -1.0 ? 1 : (x1 == 1.0 ? 2 : 0));
            }
            rs[2] = eq ? 3 : (x2 == 0.0 ? 1 : 0);
          }
          return;
        }
        // clamp kind of this block (q2 shift already folded in by the assembly kernel)
        const bool contact = ((pk >> 20) & 1u) == KIND_CONTACT;
        double lo01 = contact ? -1.0 : -kInf, hi01 = contact ? 1.0 : kInf;
        const double lo2 = contact ? 0.0 : -kInf;
        if (COULOMB && contact) {
          const double bnd = mu * (x2 > 0.0 ? x2 : 0.0);
          lo01 = -bnd; hi01 = bnd;
        }
        double n0 = x0 + e0 * IA0;
        unsigned long long flags = 0ull;
        if (COULOMB) flags = (n0 < lo01) ? 1ull : ((n0 > hi01) ? 2ull : 0ull);
        n0 = clamp_sel(n0, lo01, hi01);
        d0 = n0 - x0;
        double n1 = x1 + (e1 - DO0 * d0) * IA1;
        if (COULOMB) flags |= ((n1 < lo01) ? 1ull : ((n1 > hi01) ? 2ull : 0ull)) << 2;
        n1 = clamp_sel(n1, lo01, hi01);
        d1 = n1 - x1;
        double n2 = x2 + ((e2 - DO1 * d0) - DO2 * d1) * IA2;
        n2 = (n2 < lo2) ? lo2 : n2;
        d2 = n2 - x2;
        const unsigned long long pk_out = COULOMB ? ((pk_lam & ~(15ull << PK_FLAGS)) | (flags << PK_FLAGS)) : pk_lam;
        st_sector(reinterpret_cast<double*>(gs + lam_off), n0, n1, n2, __longlong_as_double((long long)pk_out));
      }
      // impulse scatter: a += M^-1 J^T delta
      const double ix = RC0 * d0 + RC3 * d1 + RC6 * d2, iy = RC1 * d0 + RC4 * d1 + RC7 * d2, iz = RC2 * d0 + RC5 * d1 + RC8 * d2;
      {
        const double cx = R1Y * iz - R1Z * iy, cy = R1Z * ix - R1X * iz, cz = R1X * iy - R1Y * ix;   // r1 x imp
        double dax, day, daz;
        if (ISO) { dax = m1[1] * cx; day = m1[1] * cy; daz = m1[1] * cz; }
        else { dax = m1[1] * cx + m1[2] * cy + m1[3] * cz; day = m1[4] * cx + m1[5] * cy + m1[6] * cz; daz = m1[7] * cx + m1[8] * cy + m1[9] * cz; }
        a1a.x += m1[0] * ix; a1a.y += m1[0] * iy; a1b.x += m1[0] * iz;
        a1b.y += dax; a1c.x += day; a1c.y += daz;
        if (i1 >= 0) { q1[0] = a1a; q1[1] = a1b; q1[2] = a1c; }
      }
      {
        const double cx = R0Y * iz - R0Z * iy, cy = R0Z * ix - R0X * iz, cz = R0X * iy - R0Y * ix;   // r0 x imp
        double dax, day, daz;
        if (ISO) { dax = m0[1] * cx; day = m0[1] * cy; daz = m0[1] * cz; }
        else { dax = m0[1] * cx + m0[2] * cy + m0[3] * cz; day = m0[4] * cx + m0[5] * cy + m0[6] * cz; daz = m0[7] * cx + m0[8] * cy + m0[9] * cz; }
        a0a.x -= m0[0] * ix; a0a.y -= m0[0] * iy; a0b.x -= m0[0] * iz;
        a0b.y -= dax; a0c.x -= day; a0c.y -= daz;
        if (i0 >= 0) { q0[0] = a0a; q0[1] = a0b; q0[2] = a0c; }
      }
    };
    auto reduce4 = [&]() {
#pragma unroll
      for (int o = LPW / 2; o > 0; o >>= 1) {
        se += __shfl_xor_sync(FULL, se, o);
        s1 += __shfl_xor_sync(FULL, s1, o);
        s2 += __shfl_xor_sync(FULL, s2, o);
        s3 += __shfl_xor_sync(FULL, s3, o);
      }
    };

    if (R > 0 && __any_sync(FULL, active)) {
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
      start_rounds();
      while (true) {
        const bool probe = (phase == PH_PROBE);
        const int mode = (phase == PH_INIT) ? MODE_INIT : (phase == PH_UPDATE ? MODE_UPDATE : MODE_RESID);
        const bool on = (phase == PH_EXACT) ? need_exact : active;
        const int nsteps = probe ? 1 : R;
        unsigned roff = 0;
        double2 buf[SPIECES];
        for (int t = 0; t < nsteps; t++) {
          int start, total = 0, nxt = 0, cnt;
          const unsigned char* stage = stage0;
          if (probe) {                             // the world's own chunk, in its slice of the staging buffer
            mbar_wait(bar2, parity2);
            parity2 ^= 1u;
            start = sub * LPW;
            cnt = probe_cnt;
          } else {
            mbar_wait(bar, parity);
            parity ^= 1u;
            start = stage[sub]; total = stage[G]; nxt = stage[HDR_NEXT];
            cnt = (int)stage[sub + 1] - start;
            if (total > 32 || nxt > 32 || cnt < 0 || cnt > LPW || start + cnt > total) {   // same guard for the header
              if (sl == 0 && valid) atomicOr(&d.status[wc], 64);
              cnt = 0; total = min(total, 32); nxt = min(nxt, 32);
            }
          }
          const bool mine = on && sl < cnt;
          const unsigned cur_off = probe ? probe_off : roff;
          const int cur_meta = probe ? probe_meta : (start | (total << 8) | (cnt << 16));
          if (phase == PH_INIT && t == 0) { probe_off = 0; probe_meta = cur_meta; probe_cnt = cnt; }   // first probe: the world's stage 0
          double x0 = 0, x1 = 0, x2 = 0;
          unsigned long long pk_lam = 0ull;       // the block's packed word travels in the 4th slot of its multiplier sector
          if (mine) {
            const double2* lq = reinterpret_cast<const double2*>(stage + HDRB) + (start + sl) * 2;
            const double2* sp = reinterpret_cast<const double2*>(stage + HDRB + (probe ? 32 : total) * LAMB) + (start + sl) * SPIECES;
            const double2 la = lq[0], lb = lq[1];
            x0 = la.x; x1 = la.y; x2 = lb.x;
            pk_lam = (unsigned long long)__double_as_longlong(lb.y);
#pragma unroll
            for (int p = 0; p < SPIECES; p++) buf[p] = sp[p];
          }
          // The staging buffer is handed back to the TMA unit here.  The loads above are generic-proxy
          // reads, the next copy is an async-proxy write: the two proxies are ordered only by a
          // cross-proxy fence.  A generic fence (__threadfence_block) is NOT enough: with it (or with
          // nothing) the next round could land under loads that had not been performed yet and the
          // lanes worked on the wrong round's blocks -- rare at 4 worlds per warp, 1-2 % of the
          // worlds per step at 32 worlds per warp and >= 2 resident CTAs per SM, found with
          // tools/determinism_check.py (bit-for-bit repeatability of a full-size step) and pinned
          // down by switching the fence at run time inside one binary.
          asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
          __syncwarp();                            // staging buffer free again
          const unsigned roff_next = roff + round_bytes(total, BLKB);
          if (probe) {
            start_rounds();                        // speculate "continue": the first rounds stream in meanwhile
          } else if (t + 1 < R) {
            issue_round(roff_next, nxt);
          }
          if (!probe && pf > 0) {
            // HBM -> L2 prefetch cursor kept pf x 4 KB ahead of the consumer (one 128-byte line per
            // lane and span; the cursor wraps: the next sweep streams the same bytes again).  The
            // loaded DRAM latency is ~2-3 us (tools/micro/dram_chunk_bench), one 4 KB round per
            // warp in flight cannot cover it.
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
          step(buf, x0, x1, x2, pk_lam, mode, mine, cur_off + HDRB + (unsigned)(((cur_meta & 255) + sl) * LAMB), cur_off, cur_meta, !probe);
          __syncwarp();                            // accumulator writes visible to the next round
          roff = roff_next;
        }
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
          if (need_exact && bb > 0.0) { probe_off = bo; probe_meta = bc; probe_cnt = bc >> 16; }
          if (!__any_sync(FULL, active)) break;
          phase = PH_UPDATE;
          if (active) ++it;
          start_rounds();
          continue;
        }
        if (phase == PH_UPDATE) {
          // multipliers were written with generic stores; the async proxy reads them back next sweep
          // (.global: the multipliers live in global memory; the space-less form also emits MEMBAR.ALL.GPU)
          asm volatile("fence.proxy.async.global;" ::: "memory");
          __syncwarp();
          ++k;
        }
        // after PH_INIT (k = 0) or PH_UPDATE: start the check of x_k
        se = s1 = s2 = s3 = 0.0;
        best = -1.0;
        if (k < k_max && __any_sync(FULL, active && probe_cnt > 0)) {
          phase = PH_PROBE;
          issue_probe(active);
        } else {
          phase = PH_EXACT;
          need_exact = active;
          start_rounds();
        }
      }
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

template <bool F32>
size_t stream_smem(const EggDev& d, int lpw) {
  const int G = 32 / lpw;
  return 64 + (size_t)G * 48 * d.n + (size_t)(HDRB + 32 * ((F32 ? RECB32 : RECB64) + LAMB));   // FP64, 64 bodies: 19072 B, 11 CTAs per SM
}

template <int LPW, int MINB, int ISO, bool F32, bool COULOMB>
cudaError_t launch(const EggDev& d, double dt, const double* mu, cudaStream_t s) {
  constexpr int G = 32 / LPW;
  const size_t smem = stream_smem<F32>(d, LPW);
  // shared-memory attribute and occupancy are looked up once per (kernel instance, shared-memory
  // size, device), not on every step
  static thread_local size_t c_smem = ~(size_t)0;
  static thread_local int c_dev = -1, c_per_sm = 0, c_sms = 148;
  cudaError_t e = cudaSuccess;
  int dev = 0;
  EGG_FIRST(e, cudaGetDevice(&dev));
  if (e != cudaSuccess) return e;
  if (smem != c_smem || dev != c_dev) {
    EGG_FIRST(e, cudaFuncSetAttribute(egg_pgs_stream_kernel<LPW, MINB, ISO, F32, COULOMB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    EGG_FIRST(e, cudaDeviceGetAttribute(&c_sms, cudaDevAttrMultiProcessorCount, dev));
    EGG_FIRST(e, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&c_per_sm, egg_pgs_stream_kernel<LPW, MINB, ISO, F32, COULOMB>, 32, smem));
    if (e != cudaSuccess) return e;
    if (c_per_sm < 1) return cudaErrorLaunchOutOfResources;   // the kernel does not fit an SM with this much shared memory
    c_smem = smem; c_dev = dev;
  }
  int per_sm = c_per_sm;
  if (d.sel.ctas_per_sm > 0 && d.sel.ctas_per_sm < per_sm) per_sm = d.sel.ctas_per_sm;
  const int groups = (d.W + G - 1) / G;
  const int grid = groups < c_sms * per_sm ? groups : c_sms * per_sm;
  e = cudaMemsetAsync(d.work_ctr, 0, sizeof(int), s);
  if (e != cudaSuccess) return e;   // without the reset the persistent kernel would find an exhausted queue and do nothing
  egg_pgs_stream_kernel<LPW, MINB, ISO, F32, COULOMB><<<grid, 32, smem, s>>>(d, dt, d.sel.pf, mu);
  return cudaGetLastError();
}

// Registers are allocated per scheduler (16384 each): 12 one-warp CTAs per SM = 3 per scheduler
// = 168 registers.
template <int MINB, int ISO, bool F32, bool COULOMB>
cudaError_t launch_lpw(const EggDev& d, double dt, const double* mu, cudaStream_t s) {
  switch (d.lpw) {
    case 1: return launch<1, MINB, ISO, F32, COULOMB>(d, dt, mu, s);
    case 2: return launch<2, MINB, ISO, F32, COULOMB>(d, dt, mu, s);
    case 4: return launch<4, MINB, ISO, F32, COULOMB>(d, dt, mu, s);
    case 16: return launch<16, MINB, ISO, F32, COULOMB>(d, dt, mu, s);
    default: return launch<8, MINB, ISO, F32, COULOMB>(d, dt, mu, s);
  }
}
// One staging buffer per warp.  A second buffer (two rounds in flight) was measured no better
// anywhere -- stack10 4096 worlds 26.9 vs 26.2 ms, legged20 106 vs 90 ms, pile64 8.8 vs 8.1 ms --
// and was removed again.
template <int MINB, int ISO>
cudaError_t launch_nbuf(const EggDev& d, double dt, const double* mu, cudaStream_t s) {
  if (mu) {   // Coulomb friction (egg_set_friction): the twins of the BOX instances
    if (d.blkb == RECB32 + LAMB) return launch_lpw<MINB, ISO, true, true>(d, dt, mu, s);
    return launch_lpw<MINB, ISO, false, true>(d, dt, mu, s);
  }
  if (d.blkb == RECB32 + LAMB) return launch_lpw<MINB, ISO, true, false>(d, dt, mu, s);
  return launch_lpw<MINB, ISO, false, false>(d, dt, mu, s);
}

size_t schedule_per_world(const EggDev& d) { return ((size_t)(d.n + 4 * d.nrec + 2 + 7) & ~(size_t)7) * sizeof(unsigned short); }

}  // namespace

int egg_stream_blkb(int precision) { return (precision == 32 ? RECB32 : RECB64) + LAMB; }

size_t egg_stream_rec_bytes(int W, int nrec, int lpw) {
  const int G = 32 / lpw;
  return (size_t)((W + G - 1) / G) * group_stride_bytes(nrec, G);
}

size_t egg_stream_smem(const EggDev& d) {
  const size_t solve = (d.blkb == RECB32 + LAMB) ? stream_smem<true>(d, d.lpw) : stream_smem<false>(d, d.lpw);
  const size_t recs = (size_t)(EGG_DYN + EGG_STAT + 6) * d.n * sizeof(double);
  const size_t sched = schedule_per_world(d);
  size_t m = solve > recs ? solve : recs;
  return m > sched ? m : sched;
}

template <int NT>
cudaError_t launch_records_nt(const EggDev& d, double dt, int G, size_t smem, cudaStream_t s) {
  cudaError_t e = cudaSuccess;
  if (smem > 48 * 1024) EGG_FIRST(e, cudaFuncSetAttribute(egg_records_kernel<NT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  if (e != cudaSuccess) return e;
  egg_records_kernel<NT><<<d.W, NT, smem, s>>>(d, dt, G);
  return cudaGetLastError();
}
// Threads per world by the constraints a world typically has (joints + a few contacts per body), not
// by its capacity.  Measured (131072 x legged20, ~43 constraints): 3.8 ms at 256 threads, 1.8 at 64,
// 1.6 at 32; 16384 x pile64 (~410): 1.41 ms at 256, 1.24 at 128, 1.27 at 64.  EGG_RECORDS_NT
// (d.sel.records_nt) is rounded up to an instance: 32 / 64 / 128 / 256, or 32 / 128 / 256 for the
// record kernel of the run format (egg_pgs_runs.cu).
int egg_records_threads(const EggDev& d) {
  const int est = d.nj + 6 * d.n;
  const int nt = d.sel.records_nt ? d.sel.records_nt : (est <= 192 ? 32 : (est <= 768 ? 128 : 256));
  if (nt <= 32) return 32;
  if (nt <= 64 && d.rmax == 0) return 64;
  if (nt <= 128) return 128;
  return 256;
}

cudaError_t launch_records(const EggDev& d, double dt, int G, size_t smem, cudaStream_t s) {
  switch (egg_records_threads(d)) {
    case 32: return launch_records_nt<32>(d, dt, G, smem, s);
    case 64: return launch_records_nt<64>(d, dt, G, smem, s);
    case 128: return launch_records_nt<128>(d, dt, G, smem, s);
    default: return launch_records_nt<256>(d, dt, G, smem, s);
  }
}

// Group-stream assembly: schedule (per world) -> rounds (per group) -> records (per world).
cudaError_t egg_launch_assemble_stream(const EggDev& d, double dt, cudaStream_t s) {
  const int G = 32 / d.lpw;
  cudaError_t e = cudaSuccess;
  {
    const size_t per = schedule_per_world(d);
    int wpc = (int)((size_t)200 * 1024 / per);
    if (wpc > 4) wpc = 4;
    if (wpc < 1) wpc = 1;
    const size_t smem = wpc * per;
    if (smem > 48 * 1024) EGG_FIRST(e, cudaFuncSetAttribute(egg_schedule_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    if (e != cudaSuccess) return e;
    egg_schedule_kernel<<<(d.W + wpc - 1) / wpc, 128, smem, s>>>(d, d.rmax > 0 ? d.run_cap : d.lpw, wpc, d.rmax);
  }
  if (d.rmax > 0) return egg_launch_assemble_runs_tail(d, dt, s);   // run headers and run-format records (egg_pgs_runs.cu)
  const int ngroups = (d.W + G - 1) / G;
  egg_rounds_kernel<<<(ngroups + 3) / 4, 128, 0, s>>>(d, G);
  const size_t smem = (size_t)(EGG_DYN + EGG_STAT + 6) * d.n * sizeof(double);
  return launch_records(d, dt, G, smem, s);
}

// With a friction table the caller keeps d.rmax = 0 (egg_capi.cu): the run format has BOX friction only.
cudaError_t egg_launch_solve_pgs_stream(const EggDev& d, double dt, const double* mu, cudaStream_t s) {
  if (d.rmax > 0) return egg_launch_solve_pgs_runs(d, dt, s);
  if (d.iso == 2) return launch_nbuf<12, 2>(d, dt, mu, s);
  if (d.iso == 1) return launch_nbuf<12, 1>(d, dt, mu, s);
  return launch_nbuf<8, 0>(d, dt, mu, s);
}
