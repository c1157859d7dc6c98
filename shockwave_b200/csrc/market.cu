// market.cu — dense primal-dual price-response iteration over the allocation tensor
// X[S][J][W][T] (scenario x job x worker type x planning round, fp32, t innermost).
//
// This is the general *volatile Fisher market* form of Shockwave's relaxation: a job may progress at a
// different rate r_jw (epochs per round) on every worker type and every (type, round) slot has its own
// capacity and its own price — the formulation the reference leaves as future work ("we assume homogeneous
// hardware", scripts/drivers/simulate_scheduler_with_trace.py:76-78) and BASELINE.json's north_star
// names.  Objective (per scenario), same pieces as shockwave.py:565-568:
//     sum_j plog((c_j + P_j)/E_j)/(J T) - k max_j max(0, R_j - dbar_j P_j),   P_j = sum_wt r_jw x_jwt
//     s.t. sum_j g_j x_jwt <= G_wt  (per worker type and round),  sum_w x_jwt <= 1,  0 <= x <= 1.
// Algorithm: diagonally preconditioned primal-dual hybrid gradient (Chambolle-Pock with the Pock-Chambolle
// alpha = 1 step sizes) on the saddle form of that LP.  Duals: one price pi_wt per capacity row, the marginal
// utility m_j of every job (conjugate of the piece-wise linear log, prox by a segment scan) and the makespan
// multipliers omega_j (projection on {omega >= 0, sum omega <= k D T}).  One iteration =
//   market_step (the dense pass):  x <- proj_{box, budget}( x + tau_jt (theta_j r_jw - pi_wt g_j / G_wt) ),
//       tau_jt = 1 / (pw max_w (g_j / G_wt + r_jw beta_j)), with — fused in the same pass — the row reduction
//       P_j (warp shuffles) and the column reduction sum_j g_j x_jwt (registers -> shared memory -> one atomicAdd
//       per column and CTA).  Reads X once, writes X once: 8 bytes per element, HBM bound.
//   market_dual (O(J + W T) per scenario): dual steps on the EXTRAPOLATED reductions 2 P(x+) - P(x) (linear in x, so
//       the dense pass never needs the previous X) and the new theta_j = m_j/E_j + omega_j dbar_j/(D T).
// Two-level in time (api.cu): the same kernels first iterate on the tensor coarsened to 4 super-rounds (1/16 of the
// traffic at T = 64), the result is prolongated and the fine passes only have to absorb what differs between rounds.
// The fixed point is the LP optimum (tests/test_gpu_market.py: HiGHS LP of the heterogeneous relaxation,
// oracle/market_lp.py); on homogeneous inputs (W = 1, r_j = D/dbar_j) that is the relaxation solve.cu solves exactly.
#include <math.h>

#include "swb_common.cuh"
#include "swb_internal.h"

namespace swb {

#define MK_THREADS 256
// row sums go through global atomics when the Q = T/4 threads of a job are not a power-of-two sub-warp
#define Q_ROW_ATOMICS(T) ((((T) >> 2) > 32) || ((((T) >> 2) & (((T) >> 2) - 1)) != 0))

__device__ __forceinline__ float4 ld_stream(const float4 *p) {
  float4 v;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
  return v;
}
__device__ __forceinline__ void st_stream(float4 *p, const float4 &v) {
  asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1,%2,%3,%4};"
               :: "l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

__device__ __forceinline__ float rcp_ftz(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// One job's W x 4 block of the tensor (all worker types of four consecutive rounds) through one primal step.
//   MODE 0: x <- proj( x + tau (theta r_w - price_wt g) ),  tau = ipw / max_w (g icap_wt + r_w beta); the projection is
//           the Euclidean one on {x >= 0, sum_w x <= 1} (x <= 1 is implied), exact for W <= 4 by active-set pruning —
//           tau is the same for all types of a (job, round) so that the Euclidean projection is the right one;
//   MODE 1: x <- clamp(x cs_wt, 0, 1)   (measurement pass with cs = 1, final repair with cs = min(1, G/load)).
// ca = icap (MODE 0) or colscale (MODE 1), cb = price * icap (MODE 0).
template <int W, int MODE>
__device__ __forceinline__ void respond(float4 (&x)[W], const float (&ca)[W][4], const float (&cb)[W][4],
                                        const float (&r)[W], float theta, float beta, float gj, float ipw) {
  float v[W][4];
#pragma unroll
  for (int w = 0; w < W; ++w) { v[w][0] = x[w].x; v[w][1] = x[w].y; v[w][2] = x[w].z; v[w][3] = x[w].w; }
  if (MODE == 1) {
#pragma unroll
    for (int w = 0; w < W; ++w)
#pragma unroll
      for (int e = 0; e < 4; ++e) v[w][e] = __saturatef(v[w][e] * ca[w][e]);
  } else {
    float rb[W], gain[W];
#pragma unroll
    for (int w = 0; w < W; ++w) { rb[w] = r[w] * beta; gain[w] = theta * r[w]; }
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      float den = fmaf(gj, ca[0][e], rb[0]);
#pragma unroll
      for (int w = 1; w < W; ++w) den = fmaxf(den, fmaf(gj, ca[w][e], rb[w]));
      const float tau = ipw * rcp_ftz(den);      // den >= r beta > 0, never denormal: bare MUFU.RCP (no range fix-up)
      float y[W], pos = 0.f;
#pragma unroll
      for (int w = 0; w < W; ++w) {
        y[w] = fmaf(tau, fmaf(-cb[w][e], gj, gain[w]), v[w][e]);
        pos += fmaxf(y[w], 0.f);
      }
      if (W == 1) {
        v[0][e] = __saturatef(y[0]);
      } else if (pos <= 1.f) {
#pragma unroll
        for (int w = 0; w < W; ++w) v[w][e] = fmaxf(y[w], 0.f);
      } else {
        // simplex projection: theta = (sum_active y - 1)/|active|, prune y_w <= theta, at most W rounds
        bool act[W];
#pragma unroll
        for (int w = 0; w < W; ++w) act[w] = true;
        float th = 0.f;
#pragma unroll
        for (int it = 0; it < W; ++it) {
          float sm = 0.f, n = 0.f;
#pragma unroll
          for (int w = 0; w < W; ++w) { sm += act[w] ? y[w] : 0.f; n += act[w] ? 1.f : 0.f; }
          th = __fdividef(sm - 1.f, n);
#pragma unroll
          for (int w = 0; w < W; ++w) act[w] = act[w] && y[w] > th;
        }
#pragma unroll
        for (int w = 0; w < W; ++w) v[w][e] = fmaxf(y[w] - th, 0.f);
      }
    }
  }
#pragma unroll
  for (int w = 0; w < W; ++w) x[w] = make_float4(v[w][0], v[w][1], v[w][2], v[w][3]);
}

// Dense pass.  Grid (job tiles, S).  A thread owns one float4 of rounds (4 consecutive t) of a job and
// loops over that job's worker types, so the budget projection over w is thread-local.  Q = T/4
// threads cover a job; MK_THREADS/Q jobs per sweep; U sweeps are loaded before any is used so that
// U*W 16-byte loads per thread are in flight (the pass is HBM bound: memory-level parallelism first).
template <int W, int U, int MODE>
__global__ void __launch_bounds__(MK_THREADS) market_step_kernel(MarketLaunch L) {
  extern __shared__ float sm[];           // [W*T] icap or colscale | [W*T] price | [W*T] column accumulators
  const int s = blockIdx.y;
  const int T = L.T, J = L.J, WT = W * T;
  const int Q = T >> 2;                   // float4 groups per (job, type) row
  float *cs = sm, *pi = sm + WT, *acc = sm + 2 * WT;
  const float *cs_g = MODE == 1 ? L.colscale + (size_t)s * WT : L.icap, *pi_g = L.price + (size_t)s * WT;
  for (int i = threadIdx.x; i < WT; i += blockDim.x) { cs[i] = cs_g[i]; pi[i] = pi_g[i]; acc[i] = 0.f; }
  __syncthreads();
  const float ipw = 1.0f / L.pws[s];
  const int q = threadIdx.x % Q;          // which 4 rounds
  const int jl = threadIdx.x / Q;         // job lane within the sweep
  const int jobs_per_sweep = MK_THREADS / Q;
  const int j0 = blockIdx.x * L.jobs_per_cta;
  const int j1 = min(J, j0 + L.jobs_per_cta);
  const bool active_lane = jl < jobs_per_sweep;
  float colacc[W][4];
  float csr[W][4], pir[W][4];             // this thread's columns never change: keep them in registers
#pragma unroll
  for (int w = 0; w < W; ++w)
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      colacc[w][e] = 0.f;
      csr[w][e] = active_lane ? cs[w * T + 4 * q + e] : 1.f;
      pir[w][e] = active_lane ? pi[w * T + 4 * q + e] : 0.f;
    }
  for (int jb = j0; jb < j1; jb += U * jobs_per_sweep) {
    float4 x[U][W];
    float theta[U], beta[U], gj[U], r[U][W];
    bool live[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int j = jb + u * jobs_per_sweep + jl;
      live[u] = active_lane && j < j1;
      if (live[u]) {
        const size_t sj = (size_t)s * J + j;
        const float4 *xrow = reinterpret_cast<const float4 *>(L.X + sj * WT);
#pragma unroll
        for (int w = 0; w < W; ++w) x[u][w] = ld_stream(xrow + w * Q + q);
        const float4 jp = L.jobpack[sj];
        theta[u] = jp.x; beta[u] = jp.y; gj[u] = jp.z; r[u][0] = jp.w;
#pragma unroll
        for (int w = 1; w < W; ++w) r[u][w] = L.rate[(L.per_scn ? sj : (size_t)j) * W + w];
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int j = jb + u * jobs_per_sweep + jl;
      float rowp = 0.f;
      if (live[u]) {
        const size_t sj = (size_t)s * J + j;
        float4 *xrow = reinterpret_cast<float4 *>(L.X + sj * WT);
        respond<W, MODE>(x[u], csr, pir, r[u], theta[u], beta[u], gj[u], ipw);
#pragma unroll
        for (int w = 0; w < W; ++w) {
          const float4 y = x[u][w];
          st_stream(xrow + w * Q + q, y);
          rowp = fmaf(r[u][w], (y.x + y.y) + (y.z + y.w), rowp);
          colacc[w][0] = fmaf(gj[u], y.x, colacc[w][0]); colacc[w][1] = fmaf(gj[u], y.y, colacc[w][1]);
          colacc[w][2] = fmaf(gj[u], y.z, colacc[w][2]); colacc[w][3] = fmaf(gj[u], y.w, colacc[w][3]);
        }
      }
      // row reduction over the Q threads of the job: shuffles inside the warp when Q is a power of two
      // <= 32, else the partial sums go through global atomics (rowp is zeroed by the dual pass)
      if (!Q_ROW_ATOMICS(T)) {
        for (int o = Q >> 1; o > 0; o >>= 1) rowp += __shfl_xor_sync(SWB_FULL, rowp, o);
        if (live[u] && q == 0) L.rowp[(size_t)s * J + j] = rowp;
      } else if (live[u]) {
        atomicAdd(&L.rowp[(size_t)s * J + j], rowp);
      }
    }
  }
  // column reduction: registers -> shared -> global
  if (active_lane) {
#pragma unroll
    for (int w = 0; w < W; ++w) {
      const int c0 = w * T + 4 * q;
      atomicAdd(&acc[c0 + 0], colacc[w][0]); atomicAdd(&acc[c0 + 1], colacc[w][1]);
      atomicAdd(&acc[c0 + 2], colacc[w][2]); atomicAdd(&acc[c0 + 3], colacc[w][3]);
    }
  }
  __syncthreads();
  float *col_g = L.colload + (size_t)s * WT;
  for (int i = threadIdx.x; i < WT; i += blockDim.x) atomicAdd(&col_g[i], acc[i]);
}


// Fast path of the dense pass: rounds per job T = 4 Q with Q a power of two <= 32 fixed at compile time (T = 32 / 64 /
// 128), so the row reduction is a fixed shuffle tree, every index is a 32-bit offset from a per-scenario base pointer
// and nothing depends on T at run time.  Same arithmetic, same order of operations as market_step_kernel (the numpy
// restatement in tests/ref_market.py covers both); the generic kernel spent ~40 thread instructions per tensor element,
// 71 % issue-active, which held the pass at 0.81 of the HBM peak (ncu r02).
template <int W, int U, int Q>
__global__ void __launch_bounds__(MK_THREADS) market_step_fast(MarketLaunch L) {
  constexpr int T = 4 * Q, WT = W * T, JPS = MK_THREADS / Q;
  __shared__ float acc[WT];
  const int s = blockIdx.y, J = L.J;
  const int q = threadIdx.x & (Q - 1), jl = threadIdx.x / Q;
  const float *cs_g = L.icap, *pi_g = L.price + (size_t)s * WT;
  for (int i = threadIdx.x; i < WT; i += MK_THREADS) acc[i] = 0.f;
  const float ipw = 1.0f / L.pws[s];
  const int j0 = blockIdx.x * L.jobs_per_cta;
  const int j1 = min(J, j0 + L.jobs_per_cta);
  float colacc[W][4], csr[W][4], pir[W][4];
#pragma unroll
  for (int w = 0; w < W; ++w) {
    const float4 c4 = *reinterpret_cast<const float4 *>(cs_g + w * T + 4 * q);
    const float4 p4 = *reinterpret_cast<const float4 *>(pi_g + w * T + 4 * q);
    csr[w][0] = c4.x; csr[w][1] = c4.y; csr[w][2] = c4.z; csr[w][3] = c4.w;
    pir[w][0] = p4.x; pir[w][1] = p4.y; pir[w][2] = p4.z; pir[w][3] = p4.w;
#pragma unroll
    for (int e = 0; e < 4; ++e) colacc[w][e] = 0.f;
  }
  __syncthreads();
  const size_t sJ = (size_t)s * J;
  float4 *xs = reinterpret_cast<float4 *>(L.X + sJ * WT) + q;          // + (j W + w) Q : 32-bit offsets below
  const float4 *jpk = L.jobpack + sJ;
  float *rp = L.rowp + sJ;
  const float *rt = L.rate + (L.per_scn ? sJ * W : 0);
  for (int jb = j0 + jl; jb < j1; jb += U * JPS) {
    float4 x[U][W];
    float theta[U], beta[U], gj[U], r[U][W];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int j = jb + u * JPS;
      if (j < j1) {
#pragma unroll
        for (int w = 0; w < W; ++w) x[u][w] = ld_stream(xs + (j * W + w) * Q);
        const float4 jp = jpk[j];                  // (theta, beta, g, rate on type 0): one 16-byte load per job
        theta[u] = jp.x; beta[u] = jp.y; gj[u] = jp.z; r[u][0] = jp.w;
#pragma unroll
        for (int w = 1; w < W; ++w) r[u][w] = rt[j * W + w];
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int j = jb + u * JPS;
      const bool live = j < j1;
      float rowp = 0.f;
      if (live) {
        respond<W, 0>(x[u], csr, pir, r[u], theta[u], beta[u], gj[u], ipw);
#pragma unroll
        for (int w = 0; w < W; ++w) {
          const float4 y = x[u][w];
          st_stream(xs + (j * W + w) * Q, y);
          rowp = fmaf(r[u][w], (y.x + y.y) + (y.z + y.w), rowp);
          colacc[w][0] = fmaf(gj[u], y.x, colacc[w][0]); colacc[w][1] = fmaf(gj[u], y.y, colacc[w][1]);
          colacc[w][2] = fmaf(gj[u], y.z, colacc[w][2]); colacc[w][3] = fmaf(gj[u], y.w, colacc[w][3]);
        }
      }
#pragma unroll
      for (int o = Q >> 1; o > 0; o >>= 1) rowp += __shfl_xor_sync(SWB_FULL, rowp, o);
      if (live && q == 0) rp[j] = rowp;
    }
  }
#pragma unroll
  for (int w = 0; w < W; ++w) {
    const int c0 = w * T + 4 * q;
    atomicAdd(&acc[c0 + 0], colacc[w][0]); atomicAdd(&acc[c0 + 1], colacc[w][1]);
    atomicAdd(&acc[c0 + 2], colacc[w][2]); atomicAdd(&acc[c0 + 3], colacc[w][3]);
  }
  __syncthreads();
  float *col_g = L.colload + (size_t)s * WT;
  for (int i = threadIdx.x; i < WT; i += MK_THREADS) atomicAdd(&col_g[i], acc[i]);
}

template <int W, int U>
static bool launch_fast(const MarketLaunch &L, dim3 grid, cudaStream_t st) {
  switch (L.T) {
    case 32: market_step_fast<W, U, 8><<<grid, MK_THREADS, 0, st>>>(L); return true;
    case 64: market_step_fast<W, U, 16><<<grid, MK_THREADS, 0, st>>>(L); return true;
    case 128: market_step_fast<W, U, 32><<<grid, MK_THREADS, 0, st>>>(L); return true;
    default: return false;
  }
}

// Per-scenario small pass.  Every phase scores the X the previous dense pass wrote (objective, makespan, worst relative
// capacity violation).  phase 0: start — step-size constants, theta / prices from the duals as they are (zero or
// prolongated from the coarse level), reductions of x^0 remembered; phase 1: the dual half of one PDHG iteration on
// the extrapolated reductions 2 red(x^{k+1}) - red(x^k); phase 2: column scale factors min(1, G/load) for the final
// repair pass; phase 3: score only.
__global__ void __launch_bounds__(1024) market_dual_kernel(MarketLaunch L) {
  __shared__ double red[2 * 64];
  __shared__ Pwl P;
  const int s = blockIdx.x;
  const int J = L.J, W = L.W, T = L.T, WT = W * T;
  const swb_params &prm = L.prm[s];
  BlockRed br(red);
  if (threadIdx.x == 0) make_pwl(P, prm);
  __syncthreads();
  const double Tf = (double)L.Tfull, rs = (double)L.rscale;
  const double invJT = 1.0 / ((double)J * Tf);
  const double DT = prm.round_duration * Tf, kk = prm.k * DT;
  double welfare = 0.0, mx = 0.0, sumg = 0.0, maxKm = 0.0, mkmax = 0.0;
  const bool eg = L.utility == 1;      // Eisenberg-Gale: sum_j log(U_j) over the jobs with E_j > 0, no makespan term
  for (int j = threadIdx.x; j < J; j += blockDim.x) {
    const size_t sj = (size_t)s * J + j, ji = L.per_scn ? sj : j;
    const double Ef = L.E[ji], cf = L.c[ji];
    sumg += (double)L.g[ji];
    if (eg) {
      if (Ef > 0.0) welfare += log(fmax(rs * (double)L.rowp[sj], 1e-300));
      continue;
    }
    const double Pj = fmin(rs * (double)L.rowp[sj], Ef - cf);
    welfare += plog(P, (cf + Pj) / Ef);
    mx = fmax(mx, fmax(0.0, L.rem[ji] - L.dbar[ji] * Pj));
    double sumr = 0.0;
    for (int w = 0; w < W; ++w) sumr += (double)L.rate[ji * W + w];
    maxKm = fmax(maxKm, (double)T * rs * L.dbar[ji] / DT * sumr);
    mkmax = fmax(mkmax, L.rem[ji] / DT);
  }
  br.sum2(welfare, sumg);
  welfare *= invJT;
  mx = br.max(mx);
  maxKm = br.max(maxKm);
  mkmax = br.max(mkmax);
  // primal weight of this scenario: the caller's, raised so that the makespan multipliers can fill their budget k D T
  // within ~32 dual steps (a step moves them by sigma_m (R_j/(D T) - ...) = pw/maxKm * O(mkmax)) — without it a large
  // k needs k D T / sigma_m ~ 1e5 iterations just to build the multipliers up
  if (L.phase == 0 && threadIdx.x == 0)
    L.pws[s] = (float)fmax((double)L.pw, mkmax > 0.0 ? kk * maxKm / (32.0 * mkmax) : 0.0);
  __syncthreads();
  const double pw = (double)L.pws[s];
  if (L.phase <= 1) {
    const double sig_m = maxKm > 0.0 ? pw / maxKm : 0.0;
    double zsum = 0.0;
    for (int j = threadIdx.x; j < J; j += blockDim.x) {
      const size_t sj = (size_t)s * J + j, ji = L.per_scn ? sj : j;
      const double Ef = L.E[ji], cf = L.c[ji];
      if (eg) {
        // utility log(U_j)/(J T), U_j = rs * row sum: prox of the conjugate of -w log(u) in closed form; a job with
        // E_j <= 0 is not part of this scenario (theta stays 0, its row stays at x = 0)
        if (L.phase == 1) {
          double sumr = 0.0;
          for (int w = 0; w < W; ++w) sumr += (double)L.rate[ji * W + w];
          double m = 0.0;
          if (Ef > 0.0 && sumr > 0.0) {
            const double du = rs * (2.0 * (double)L.rowp[sj] - (double)L.rowprev[sj]);
            const double sig_u = pw / ((double)T * rs * sumr);
            const double v = du - L.mj[sj] / sig_u;
            const double ps = 0.5 * (v + sqrt(v * v + 4.0 * invJT / sig_u));
            m = L.mj[sj] - sig_u * (du - ps);
          }
          L.mj[sj] = m;
          L.om[sj] = 0.0;
        }
        L.rowprev[sj] = L.rowp[sj];
        continue;
      }
      const double aE = rs / Ef, fD = rs * L.dbar[ji] / DT;
      if (L.phase == 1) {
        double sumr = 0.0;
        for (int w = 0; w < W; ++w) sumr += (double)L.rate[ji * W + w];
        const double Pbar = 2.0 * (double)L.rowp[sj] - (double)L.rowprev[sj];      // extrapolated, in rate units
        const double du = aE * Pbar, sig_u = pw / ((double)T * aE * sumr);
        const double capu = (Ef - cf) / Ef, u0 = cf / Ef;
        double m = L.mj[sj];
        const double v = du - m / sig_u;
        double ps = capu;
        for (int b = 0; b + 1 < P.B; ++b) {           // prox of the conjugate of the PWL log: first segment that holds it
          const double hi = fmin(fmax(P.base[b + 1] - u0, 0.0), capu);
          const double cand = v + P.slope[b] * invJT / sig_u;
          if (cand <= hi) { ps = fmax(cand, fmin(fmax(P.base[b] - u0, 0.0), capu)); break; }
        }
        m -= sig_u * (du - ps);
        L.mj[sj] = m;
        const double z = fmax(0.0, L.om[sj] + sig_m * (L.rem[ji] / DT - fD * Pbar));
        L.om[sj] = z;
        zsum += z;
      }
      L.rowprev[sj] = L.rowp[sj];
    }
    if (L.phase == 1 && !eg) {
      // projection of the makespan multipliers on {omega >= 0, sum omega <= k D T}: threshold by active-set pruning
      zsum = br.sum(zsum);
      double th = 0.0;
      if (kk <= 0.0) {
        th = 1e300;
      } else if (zsum > kk) {
        th = -1.0;
        for (int it = 0; it < 64; ++it) {
          double sm = 0.0, cn = 0.0;
          for (int j = threadIdx.x; j < J; j += blockDim.x) {
            const double z = L.om[(size_t)s * J + j];
            if (z > th) { sm += z; cn += 1.0; }
          }
          br.sum2(sm, cn);
          const double nt = (sm - kk) / fmax(cn, 1.0);
          if (!(nt > th)) break;
          th = nt;
        }
      }
      if (th > 0.0)
        for (int j = threadIdx.x; j < J; j += blockDim.x) {
          const size_t sj = (size_t)s * J + j;
          L.om[sj] = fmax(L.om[sj] - th, 0.0);
        }
    }
    for (int j = threadIdx.x; j < J; j += blockDim.x) {
      const size_t sj = (size_t)s * J + j, ji = L.per_scn ? sj : j;
      const double aE = eg ? rs : rs / L.E[ji], fD = eg ? 0.0 : rs * L.dbar[ji] / DT;
      L.jobpack[sj] = make_float4((float)(L.mj[sj] * aE + L.om[sj] * fD), (float)(aE + fD), (float)L.g[ji],
                                  L.rate[ji * W]);
      if (Q_ROW_ATOMICS(T)) L.rowp[sj] = 0.f;
    }
  } else if (Q_ROW_ATOMICS(T) && L.phase == 2) {
    for (int j = threadIdx.x; j < J; j += blockDim.x) L.rowp[(size_t)s * J + j] = 0.f;
  }
  double viol = 0.0;
  for (int i = threadIdx.x; i < WT; i += blockDim.x) {
    const size_t si = (size_t)s * WT + i;
    const double ic = (double)L.icap[i];
    const double load = (double)(L.phase >= 2 ? L.colprev[si] + L.colload[si] : L.colload[si]);
    viol = fmax(viol, load * ic - 1.0);
    if (L.phase <= 1) {
      double pi = L.pi[si];
      if (L.phase == 1) {
        const double lbar = (2.0 * load - (double)L.colprev[si]) * ic;
        pi = fmax(0.0, pi + pw / (sumg * ic) * (lbar - 1.0));
        L.pi[si] = pi;
      }
      L.price[si] = (float)(pi * ic);
      L.colprev[si] = (float)load;
      L.colload[si] = 0.f;
    } else if (L.phase == 2) {
      L.colscale[si] = (load * ic > 1.0 && load > 0.0) ? (float)(1.0 / (load * ic)) : 1.f;
      L.colprev[si] = 0.f;
      L.colload[si] = 0.f;
    }
  }
  viol = br.max(viol);
  if (threadIdx.x == 0) { L.obj[3 * s] = welfare - prm.k * mx; L.obj[3 * s + 1] = mx; L.obj[3 * s + 2] = viol; }
}

// coarse -> fine in time: X[s][j][w][t] = Xc[s][j][w][t / grp], pi[s][w][t] = pic[s][w][t / grp] / grp (a coarse
// capacity row stands for grp fine rows)
__global__ void market_prolong_kernel(const float *Xc, float *X, const double *pic, double *pi, size_t rows, int S, int W,
                                      int T, int grp) {
  const size_t n4 = rows * (size_t)(T >> 2);
  const int Tc = T / grp;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n4; i += (size_t)gridDim.x * blockDim.x) {
    const size_t row = i / (T >> 2);
    const int t0 = (int)(i % (T >> 2)) * 4;
    const float *xc = Xc + row * Tc;
    reinterpret_cast<float4 *>(X)[i] = make_float4(xc[t0 / grp], xc[(t0 + 1) / grp], xc[(t0 + 2) / grp], xc[(t0 + 3) / grp]);
  }
  const size_t np = (size_t)S * W * T;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < np; i += (size_t)gridDim.x * blockDim.x) {
    const size_t sw = i / T;
    pi[i] = pic[sw * Tc + (i % T) / grp] / (double)grp;
  }
}
// fine -> coarse (warm start from a caller's X): mean over each group of rounds
__global__ void market_restrict_kernel(const float *X, float *Xc, size_t rows, int T, int grp) {
  const int Tc = T / grp;
  const size_t n = rows * Tc;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const float *x = X + (i / Tc) * T + (i % Tc) * grp;
    float a = 0.f;
    for (int t = 0; t < grp; ++t) a += x[t];
    Xc[i] = a / (float)grp;
  }
}
__global__ void market_fill_kernel(float *p, size_t n, float v) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) p[i] = v;
}

cudaError_t launch_market_prolong(const float *Xc, float *X, const double *pic, double *pi, size_t rows, int S, int W,
                                  int T, int grp, cudaStream_t st) {
  market_prolong_kernel<<<592, 256, 0, st>>>(Xc, X, pic, pi, rows, S, W, T, grp);
  return cudaGetLastError();
}
cudaError_t launch_market_restrict(const float *X, float *Xc, size_t rows, int T, int grp, cudaStream_t st) {
  market_restrict_kernel<<<592, 256, 0, st>>>(X, Xc, rows, T, grp);
  return cudaGetLastError();
}
cudaError_t launch_market_fill(float *p, size_t n, float v, cudaStream_t st) {
  market_fill_kernel<<<148, 256, 0, st>>>(p, n, v);
  return cudaGetLastError();
}

template <int MODE>
static cudaError_t launch_generic(const MarketLaunch &L, dim3 grid, size_t smem, cudaStream_t st) {
  switch (L.W) {
    case 1: market_step_kernel<1, 4, MODE><<<grid, MK_THREADS, smem, st>>>(L); break;
    case 2: market_step_kernel<2, 4, MODE><<<grid, MK_THREADS, smem, st>>>(L); break;
    case 3: market_step_kernel<3, 2, MODE><<<grid, MK_THREADS, smem, st>>>(L); break;
    default: market_step_kernel<4, 2, MODE><<<grid, MK_THREADS, smem, st>>>(L); break;
  }
  return cudaGetLastError();
}

// dense = false: the dual pass (L.phase); dense = true: the dense pass (L.mode 0 = primal step, 1 = column scaling)
cudaError_t launch_market_iter(const MarketLaunch &L, cudaStream_t st, bool dense) {
  if (!dense) {
    market_dual_kernel<<<L.S, 1024, 0, st>>>(L);
    return cudaGetLastError();
  }
  dim3 grid((L.J + L.jobs_per_cta - 1) / L.jobs_per_cta, L.S);
  const size_t smem = 3 * (size_t)L.W * L.T * sizeof(float);
  if (L.mode == 1) return launch_generic<1>(L, grid, smem, st);
  // fast path: T in {32, 64, 128} and a scenario's slice of X addressable with 32-bit float4 offsets
  if ((size_t)L.J * L.W * (L.T / 4) < (1u << 30)) {
    bool done = false;
    switch (L.W) {
      case 1: done = launch_fast<1, 4>(L, grid, st); break;
      case 2: done = launch_fast<2, 4>(L, grid, st); break;
      case 3: done = launch_fast<3, 2>(L, grid, st); break;
      default: done = launch_fast<4, 2>(L, grid, st); break;
    }
    if (done) return cudaGetLastError();
  }
  return launch_generic<0>(L, grid, smem, st);
}

}  // namespace swb
