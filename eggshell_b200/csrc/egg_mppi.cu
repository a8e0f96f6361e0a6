// MPPI (model predictive path integral): the two data-heavy steps of the sampling planner, next to
// the step.  egg_sample_controls writes W perturbed copies of a nominal control schedule;
// egg_mppi_reduce sums them weighted by exp(-(J - J_min) / lambda).  Both touch the whole
// [H][W][c] schedule and nothing else of size: c = 6 n body-wrench components per world (6.3 GB at
// 131072 legged20 worlds and H = 50), or m actuator values with an actuator table (57 for the joint
// motors of legged20: 3.0 GB).  Every kernel here works on rows of either width.
// CEM (cross-entropy method) shares the sampler with a per-step sigma (egg_sample_controls_std) and
// refits on the elites: egg_gather_controls copies their schedules, egg_control_moments averages them.
#include "egg_internal.cuh"
#include <curand_philox4x32_x.h>   // header-only device code of the toolkit: curand_Philox4x32_10

// Two Philox words -> a uniform in (0, 1]: the top 53 bits of (lo | hi << 32), offset by 2^-54 so
// that 0 never occurs (ln u is finite, |eps| <= 8.7).  Above 0.5 the sum is a tie that rounds to
// even, so 1.0 can occur; it is harmless (ln 1 = 0 gives r = 0, sincospi(2) is finite).
__device__ __forceinline__ double egg_u01(unsigned lo, unsigned hi) {
  const unsigned long long x = ((unsigned long long)hi << 32) | lo;
  return (double)(x >> 11) * 0x1p-53 + 0x1p-54;
}

// clamp that lets NaN through (fmin/fmax would replace it by a bound)
__device__ __forceinline__ double egg_clamp(double v, double lo, double hi) { return v < lo ? lo : (v > hi ? hi : v); }

// Where the sampler kernel reads sigma.sigma from: the sampler's row [c], the same for every step
// (egg_sample_controls), or the caller's per-step [H][c] device array read like u_nom
// (egg_sample_controls_std).  Everything else, the noise included, is the same code.
enum EggSigmaFrom { EGG_SIGMA_PER_BODY, EGG_SIGMA_PER_STEP };

// Two adjacent doubles of a control row: one 16-byte access when the row width c is even (every
// pair then starts 16-byte aligned), 8-byte ones when it is odd; half: the pair is the last of an odd
// row and has no second element (read as 0).
template <bool kOdd>
__device__ __forceinline__ double2 egg_load2(const double* p, bool half) {
  if constexpr (kOdd) return make_double2(p[0], half ? 0.0 : p[1]);
  else return *reinterpret_cast<const double2*>(p);
}

// One thread per (step, world, component pair) of a control row of width c with P = ceil(c / 2) pairs:
// i = w P + p within step t, so thread i writes the elements (2p, 2p + 1) of u[t][w] and, for even c,
// a warp writes 512 consecutive bytes with 16-byte stores.  The Philox counter is q = t P + p; for
// c = 6 n this is (t n + b) 3 + p' of the body-wrench space (p = 3 b + p').  For odd c the last pair
// discards its second normal.  The noise is computed for every element whatever sigma is (sigma = 0
// costs what sigma > 0 does); global world 0 and sigma = 0 keep u_nom bit for bit (-0.0 included).
template <EggSigmaFrom kFrom, bool kOdd>
__global__ void __launch_bounds__(256) egg_mppi_sample_kernel(const double* __restrict__ u_nom, EggSampler sm, int W, int c,
                                                              int H, unsigned per_step, uint2 key, uint2 iter, int first,
                                                              double* __restrict__ u) {
  const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= per_step) return;
  const unsigned P = ((unsigned)c + 1u) >> 1;
  const unsigned p = i % P, w = i / P;
  const unsigned g = (unsigned)first + w;
  const int j = 2 * (int)p;
  const bool half = kOdd && j + 1 == c;
  const int j1 = half ? j : j + 1;   // the bounds of a missing second element are never used
  double s0 = 0.0, s1 = 0.0;
  if constexpr (kFrom == EGG_SIGMA_PER_BODY) s0 = sm.sigma[j], s1 = sm.sigma[j1];
  const double lo0 = sm.lo[j], lo1 = sm.lo[j1];
  const double hi0 = sm.hi[j], hi1 = sm.hi[j1];
  for (int t = blockIdx.y; t < H; t += gridDim.y) {
    const uint4 r = curand_Philox4x32_10(make_uint4((unsigned)t * P + p, g, iter.x, iter.y), key);
    const double u1 = egg_u01(r.x, r.y), u2 = egg_u01(r.z, r.w);
    const double rad = sqrt(-2.0 * log(u1));
    double sn, cs;
    sincospi(2.0 * u2, &sn, &cs);
    const double2 m = egg_load2<kOdd>(u_nom + (size_t)t * c + j, half);
    if constexpr (kFrom == EGG_SIGMA_PER_STEP) {
      const double2 sd = egg_load2<kOdd>(sm.sigma + (size_t)t * c + j, half);
      s0 = sd.x, s1 = sd.y;
    }
    double v0 = m.x + s0 * (rad * cs), v1 = m.y + s1 * (rad * sn);
    if (g == 0 || s0 == 0.0) v0 = m.x;
    if (g == 0 || s1 == 0.0) v1 = m.y;
    double* out = u + ((size_t)t * W + w) * c + j;
    if constexpr (kOdd) {
      out[0] = egg_clamp(v0, lo0, hi0);
      if (!half) out[1] = egg_clamp(v1, lo1, hi1);
    } else {
      *reinterpret_cast<double2*>(out) = make_double2(egg_clamp(v0, lo0, hi0), egg_clamp(v1, lo1, hi1));
    }
  }
}

// Worlds per stage-1 partial of the reduction (= the block size of its kernel).
#define EGG_MPPI_CHUNK 256

// Stage 1: block (x, y) sums the worlds [y CHUNK, (y + 1) CHUNK) of columns x*256 ... of the
// [H c + 2]-column table (u[t][w] flattened over (t, row element), then omega, then omega^2), in world
// order.  The chunk's weights are computed once into shared memory.  For a fixed world the 256
// threads read 256 consecutive doubles of u, so the loads are coalesced; each thread walks down its
// column.  A zero weight contributes exactly nothing (a NaN control of a discarded world included).
__global__ void __launch_bounds__(EGG_MPPI_CHUNK) egg_mppi_reduce_kernel(const double* __restrict__ u, int W, int c, int L,
                                                                        const double* __restrict__ cost,
                                                                        const double* __restrict__ baseline, double lambda,
                                                                        double* __restrict__ partial) {
  __shared__ double om[EGG_MPPI_CHUNK];
  const int w0 = blockIdx.y * EGG_MPPI_CHUNK;
  const int nw = min(EGG_MPPI_CHUNK, W - w0);
  const double base = *baseline;
  double o = 0.0;
  if ((int)threadIdx.x < nw) {
    const double J = cost[w0 + threadIdx.x];
    if (isfinite(J) && isfinite(base)) o = exp(-(J - base) / lambda);
  }
  om[threadIdx.x] = o;
  __syncthreads();
  const int col = blockIdx.x * blockDim.x + threadIdx.x;
  if (col >= L + 2) return;
  double s = 0.0;
  if (col < L) {
    const int t = col / c, e = col - t * c;
    const double* x = u + ((size_t)t * W + w0) * c + e;
#pragma unroll 8
    for (int k = 0; k < nw; k++) {
      const double ok = om[k], xk = x[(size_t)k * c];
      s += ok != 0.0 ? ok * xk : 0.0;
    }
  } else if (col == L) {
    for (int k = 0; k < nw; k++) s += om[k];
  } else {
    for (int k = 0; k < nw; k++) s += om[k] * om[k];
  }
  partial[(size_t)blockIdx.y * (L + 2) + col] = s;
}

// Stage 2: out[col] = the chunk partials of column col added in chunk order.
__global__ void __launch_bounds__(256) egg_mppi_reduce_final_kernel(const double* __restrict__ partial, int chunks, int L2,
                                                                    double* __restrict__ out) {
  const int col = blockIdx.x * blockDim.x + threadIdx.x;
  if (col >= L2) return;
  double s = 0.0;
#pragma unroll 8
  for (int c = 0; c < chunks; c++) s += partial[(size_t)c * L2 + col];
  out[col] = s;
}

// CEM refit (egg_control_moments): one thread per column of rows [k][L], two passes down the column
// in row order: mean = sum / k, then std = sqrt(sum (x - mean)^2 / k).  The square is rounded before
// it is added (no fused multiply-add), so the result is the plain float64 definition bit for bit and
// depends only on k, L and the rows.  Consecutive threads read consecutive doubles of a row.
__global__ void __launch_bounds__(256) egg_control_moments_kernel(const double* __restrict__ rows, int k, int L,
                                                                  double* __restrict__ out) {
  const int col = blockIdx.x * blockDim.x + threadIdx.x;
  if (col >= L) return;
  const double* x = rows + col;
  double s = 0.0;
  for (int i = 0; i < k; i++) s += x[(size_t)i * L];
  const double mean = s / k;
  double q = 0.0;
  for (int i = 0; i < k; i++) {
    const double dv = x[(size_t)i * L] - mean;
    q += __dmul_rn(dv, dv);
  }
  out[col] = mean;
  out[L + col] = sqrt(q / k);
}

// out[i][t][:] = u[t][worlds[i]][:], the c doubles of a step's row copied as they are (one thread each).
__global__ void __launch_bounds__(256) egg_gather_controls_kernel(const double* __restrict__ u, int W, int c, int H,
                                                                  const int* __restrict__ worlds, int k,
                                                                  double* __restrict__ out) {
  const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (gid >= (long long)k * H * c) return;
  const int e = (int)(gid % c);
  const long long r = gid / c;
  const int t = (int)(r % H), i = (int)(r / H);
  out[gid] = u[((size_t)t * W + worlds[i]) * c + e];
}

template <EggSigmaFrom kFrom, bool kOdd>
static cudaError_t launch_sample(const EggDev& d, int c, const EggSampler& sm, const double* u_nom, int horizon, unsigned long long seed,
                                 unsigned long long iteration, int first, double* u, cudaStream_t s) {
  const unsigned per_step = (unsigned)d.W * (((unsigned)c + 1u) >> 1);
  const dim3 grid((per_step + 255) / 256, (unsigned)min(horizon, 65535));
  egg_mppi_sample_kernel<kFrom, kOdd><<<grid, 256, 0, s>>>(u_nom, sm, d.W, c, horizon, per_step,
                                                           make_uint2((unsigned)seed, (unsigned)(seed >> 32)),
                                                           make_uint2((unsigned)iteration, (unsigned)(iteration >> 32)), first, u);
  return cudaGetLastError();
}

cudaError_t egg_launch_sample(const EggDev& d, int c, const EggSampler& sm, const double* mean, const double* std_dev, int horizon,
                              unsigned long long seed, unsigned long long iteration, int first, double* u, cudaStream_t s) {
  const EggSampler per_step{std_dev, sm.lo, sm.hi};
  if (c & 1) {
    if (!std_dev) return launch_sample<EGG_SIGMA_PER_BODY, true>(d, c, sm, mean, horizon, seed, iteration, first, u, s);
    return launch_sample<EGG_SIGMA_PER_STEP, true>(d, c, per_step, mean, horizon, seed, iteration, first, u, s);
  }
  if (!std_dev) return launch_sample<EGG_SIGMA_PER_BODY, false>(d, c, sm, mean, horizon, seed, iteration, first, u, s);
  return launch_sample<EGG_SIGMA_PER_STEP, false>(d, c, per_step, mean, horizon, seed, iteration, first, u, s);
}

cudaError_t egg_launch_gather_controls(const EggDev& d, int c, const double* u, int horizon, const int* worlds, int k, double* out,
                                       cudaStream_t s) {
  const long long total = (long long)k * horizon * c;
  egg_gather_controls_kernel<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(u, d.W, c, horizon, worlds, k, out);
  return cudaGetLastError();
}

cudaError_t egg_launch_control_moments(const double* rows, int k, int L, double* out, cudaStream_t s) {
  egg_control_moments_kernel<<<(unsigned)((L + 255) / 256), 256, 0, s>>>(rows, k, L, out);
  return cudaGetLastError();
}

int egg_mppi_chunks(int W) { return (W + EGG_MPPI_CHUNK - 1) / EGG_MPPI_CHUNK; }

cudaError_t egg_launch_mppi_reduce(const EggDev& d, int c, const double* u, int horizon, const double* cost, const double* baseline,
                                   double lambda, double* partial, double* out, cudaStream_t s) {
  const int L = horizon * c, chunks = egg_mppi_chunks(d.W);
  egg_mppi_reduce_kernel<<<dim3((unsigned)(L + 2 + EGG_MPPI_CHUNK - 1) / EGG_MPPI_CHUNK, (unsigned)chunks), EGG_MPPI_CHUNK, 0, s>>>(
      u, d.W, c, L, cost, baseline, lambda, partial);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  egg_mppi_reduce_final_kernel<<<(unsigned)(L + 2 + 255) / 256, 256, 0, s>>>(partial, chunks, L + 2, out);
  return cudaGetLastError();
}
