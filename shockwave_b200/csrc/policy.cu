// policy.cu — Gavel policies' get_allocation() on the GPU for a pooled (homogeneous) worker pool.
//
// Replaces the cvxpy -> ECOS / Gurobi LP solves of
//   MaxMinFairnessPolicy[WithPerf]        scheduler/policies/max_min_fairness.py:53-113
//   FinishTimeFairnessPolicy[WithPerf]    scheduler/policies/finish_time_fairness.py:66-157
//   MinTotalDurationPolicy[WithPerf]      scheduler/policies/min_total_duration.py:55-135
//   ThroughputNormalizedByCostSumWithPerfSLOs (MST)  scheduler/policies/max_sum_throughput.py:49-108
// for the case every worker type with capacity has the same throughput per job (always true for the
// non-Perf wrappers, which overwrite the matrix with the v100 column / with 1.0, and for Shockwave's
// homogeneous clusters, scheduler/scheduler.py:1128).  With one pooled type of N workers the base
// constraints (policy.py:58-65) read  0 <= x_j <= 1,  sum_j sf_j x_j <= N  and every one of these LPs
// has a closed form or a monotone 1-D search, evaluated here with block reductions in float64.
// The host splits x_j over the real worker types in proportion to their capacities.
#include <math.h>

#include "swb_common.cuh"
#include "swb_internal.h"

namespace swb {

// ---- which optimal x: the interior-point selection -------------------------------------------------------
// These LPs are degenerate in x.  The reference solves them with interior-point codes (ECOS; Gurobi barrier for the
// finish-time-fairness cone program, utils.py:603-685) whose iterates converge to the ANALYTIC CENTRE of the optimal
// face, and the closed loop is sensitive to that choice (a simplex vertex with the same objective moves the avg JCT of
// the canonical trace by 6 %; the centre reproduces the golden pickles within 0.8 %, tests/golden/tacc32_policy_pins.json).
// Pooled form (definition and numpy restatement: oracle/gavel_lp.py:analytic_centre_box):
//     maximise  sum_j [ w_lo log(x_j - lo_j) + w_x log x_j + log(1 - x_j) ] + log(N - sum_j sf_j x_j)
// On entry L.x holds lo_j (the job's requirement at the optimal scalar); on exit the centre.  Stationarity gives
// x_j(lam) as the root of a decreasing function (safeguarded Newton per job) and lam (N - sum sf x(lam)) = 1, which is
// monotone in lam (log-space bisection, one block reduction per step).
#define POL_MAXJ_PER_THREAD 8
__device__ void analytic_centre_box(const PolicyLaunch &L, BlockRed &br, double w_lo, double w_x) {
  const int J = L.J;
  const double N = L.N;
  double lo[POL_MAXJ_PER_THREAD], xs[POL_MAXJ_PER_THREAD], sfj[POL_MAXJ_PER_THREAD];
  double used0 = 0.0, usedfix = 0.0;
  int cnt = 0;
  for (int j = threadIdx.x; j < J; j += blockDim.x, ++cnt) {
    const double l = fmin(L.x[j], 1.0);
    sfj[cnt] = L.sf[j];
    const bool fixed = l >= 1.0 - 1e-15;
    lo[cnt] = fixed ? 2.0 : fmax(l, 0.0);            // 2.0 marks "fixed at 1"
    xs[cnt] = fixed ? 1.0 : fmax(l, 0.0);
    used0 += sfj[cnt] * xs[cnt];
    if (fixed) usedfix += sfj[cnt];
  }
  br.sum2(used0, usedfix);
  if (N - used0 <= 1e-12 * N) {                       // capacity is active on the whole face: x = lo is the only point
    cnt = 0;
    for (int j = threadIdx.x; j < J; j += blockDim.x, ++cnt) L.x[j] = xs[cnt];
    return;
  }
  const double Nf = N - usedfix;
  double nfree = 0.0;
  for (int q = 0; q < cnt; ++q) if (lo[q] < 2.0) { xs[q] = 0.5 * (lo[q] + 1.0); nfree += 1.0; }
  nfree = br.sum(nfree);
  // bracket of the multiplier: slack(lam) <= S = N - used0 gives lam >= 1/S; multiplying the stationarity condition
  // of job j by (x_j - lo_j) and summing gives lam (S - slack) <= nfree (w_lo + w_x), i.e. lam <= (nfree (w_lo + w_x) + 1)/S.
  // G(lam) = lam * slack(lam) - 1 is increasing: Illinois (regula falsi) with a geometric-bisection safeguard.
  const double S = N - used0;
  double a = 1.0 / S, b = (nfree * (w_lo + w_x) + 1.0) / S * (1.0 + 1e-9);
  double Ga = -1.0, Gb = 1.0;          // signs only until both ends have been evaluated
  bool have_a = false, have_b = false;
  int last = 0;
  double lam = sqrt(a * b);
  for (int it = 0; it < 80; ++it) {
    double load = 0.0;
    for (int q = 0; q < cnt; ++q) {
      if (lo[q] >= 2.0) continue;
      const double l0 = lo[q], ls = lam * sfj[q];
      double l = l0, h = 1.0, x = xs[q];
      for (int k = 0; k < 80; ++k) {
        const double d0 = x - l0, d1 = 1.0 - x;
        const double f = w_x / x - 1.0 / d1 + w_lo / d0 - ls;
        if (f == 0.0) break;
        if (f > 0.0) l = x; else h = x;
        const double fp = w_x / (x * x) + 1.0 / (d1 * d1) + w_lo / (d0 * d0);    // = -f'
        double xn = x + f / fp;
        if (xn == x) break;                                  // the Newton step is below one ulp: converged
        if (!(xn > l && xn < h)) xn = 0.5 * (l + h);
        const bool done = fabs(xn - x) <= 2e-15 * xn;
        x = xn;
        if (done) break;
      }
      xs[q] = x;
      load += sfj[q] * x;
    }
    load = br.sum(load);
    const double Gl = lam * (Nf - load) - 1.0;
    if (Gl > 0.0) {
      if (last == 1 && have_a) Ga *= 0.5;  // Illinois: an end that survives twice in a row gets half its weight
      b = lam; Gb = Gl; have_b = true; last = 1;
    } else {
      if (last == -1 && have_b) Gb *= 0.5;
      a = lam; Ga = Gl; have_a = true; last = -1;
    }
    if (b - a <= 1e-13 * b || fabs(Gl) <= 1e-13) break;
    double nl = (have_a && have_b) ? a - Ga * (b - a) / (Gb - Ga) : sqrt(a * b);
    if (!(nl > a && nl < b)) nl = sqrt(a * b);
    lam = nl;
  }
  cnt = 0;
  for (int j = threadIdx.x; j < J; j += blockDim.x, ++cnt) L.x[j] = xs[cnt];
}

__global__ void __launch_bounds__(1024, 1) policy_kernel(PolicyLaunch L) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double *red = reinterpret_cast<double *>(smem_raw);
  BlockRed br(red);
  const int J = L.J;
  const double N = L.N;
  double obj = 0.0;
  int status = 0;

  if (L.mode == SWB_POL_MAXMIN) {
    // max z : coef_j x_j >= z   ->  z = min(min_j coef_j, N / sum_j sf_j/coef_j),  x_j = z/coef_j
    double mn = 1e300, s = 0.0;
    for (int j = threadIdx.x; j < J; j += blockDim.x) {
      const double c = L.coef[j];
      mn = fmin(mn, c);
      s += L.sf[j] / c;
    }
    mn = br.min(mn);
    s = br.sum(s);
    const double z = fmin(mn, N / s);
    for (int j = threadIdx.x; j < J; j += blockDim.x) L.x[j] = fmin(1.0, z / L.coef[j]);
    __syncthreads();
    analytic_centre_box(L, br, 1.0, 1.0);
    obj = z;
  } else if (L.mode == SWB_POL_FTF) {
    // min rho : (t_j + n_j/(thr_j x_j)) / den_j <= rho   ->  x_j(rho) = n_j / (thr_j (rho den_j - t_j))
    // feasible(rho) <=> every rho den_j > t_j, x_j <= 1, sum sf_j x_j <= N ; monotone in rho
    double lo = 0.0, hi = 1.0;
    auto feasible = [&](double rho, bool write) -> bool {
      double used = 0.0, bad = 0.0;
      for (int j = threadIdx.x; j < J; j += blockDim.x) {
        const double room = rho * L.den[j] - L.t[j];
        double xj = 2.0;
        if (room > 0.0) xj = L.n[j] / (L.coef[j] * room);
        if (xj > 1.0 + 1e-12) bad += 1.0;
        used += L.sf[j] * fmin(xj, 1.0);
        if (write) L.x[j] = fmin(xj, 1.0);
      }
      br.sum2(used, bad);
      return bad == 0.0 && used <= N * (1.0 + 1e-12);
    };
    int it = 0;
    while (!feasible(hi, false) && it < 200) { lo = hi; hi *= 2.0; ++it; }
    if (it >= 200) status = 1;
    for (it = 0; it < 200 && hi - lo > 1e-13 * hi; ++it) {
      const double mid = 0.5 * (lo + hi);
      if (feasible(mid, false)) hi = mid; else lo = mid;
    }
    feasible(hi, true);
    __syncthreads();
    // cone program: t_j + n_j inv_pos(thr_j x_j) <= rho den_j -> barrier 2 log(x - lo) - log x, see gavel_lp.py
    if (status == 0) analytic_centre_box(L, br, 2.0, 0.0);
    obj = hi;
  } else if (L.mode == SWB_POL_MTD) {
    // the reference's own bisection on T (min_total_duration.py:105-131), LP feasibility in closed form
    auto feasible = [&](double T, bool write) -> bool {
      double used = 0.0, bad = 0.0;
      for (int j = threadIdx.x; j < J; j += blockDim.x) {
        const double xj = L.n[j] / (T * L.coef[j]);
        if (xj > 1.0 + 1e-12) bad += 1.0;
        used += L.sf[j] * fmin(xj, 1.0);
        if (write) L.x[j] = fmin(xj, 1.0);
      }
      br.sum2(used, bad);
      return bad == 0.0 && used <= N * (1.0 + 1e-12);
    };
    double max_T = 1000000.0, min_T = 100.0, last_max_T = max_T, best = -1.0;
    for (int outer = 0; outer < 40 && best < 0.0; ++outer) {
      while (1.05 * min_T < max_T) {
        const double T = (min_T + max_T) / 2.0;
        if (feasible(T, false)) { best = T; max_T = T; } else min_T = T;
      }
      max_T = last_max_T * 10.0;
      min_T = last_max_T;
      last_max_T *= 10.0;
    }
    if (best < 0.0) { status = 1; best = max_T; }
    feasible(best, true);
    __syncthreads();
    if (status == 0) analytic_centre_box(L, br, 1.0, 1.0);
    obj = best;
  } else if (L.mode == SWB_POL_MAXSUM) {
    // max sum_j v_j x_j : fractional knapsack by v_j/sf_j (coef = v_j), stable by job index
    int npad = 64;
    while (npad < J) npad <<= 1;
    unsigned long long *key = reinterpret_cast<unsigned long long *>(smem_raw + 2 * 64 * sizeof(double));
    unsigned short *idx = reinterpret_cast<unsigned short *>(key + npad);
    for (int i = threadIdx.x; i < npad; i += blockDim.x) {
      key[i] = i < J ? order_key(L.coef[i] / L.sf[i]) : 0ull;
      idx[i] = (unsigned short)(i < J ? i : 0xffff);
    }
    __syncthreads();
    for (int k = 2; k <= npad; k <<= 1)
      for (int j = k >> 1; j > 0; j >>= 1) {
        for (int i = threadIdx.x; i < npad; i += blockDim.x) {
          const int p = i ^ j;
          if (p > i) {
            const unsigned long long a = key[i], b = key[p];
            const unsigned short ia = idx[i], ib = idx[p];
            const bool a_first = (a > b) || (a == b && ia < ib);
            if (((i & k) == 0) != a_first) { key[i] = b; key[p] = a; idx[i] = ib; idx[p] = ia; }
          }
        }
        __syncthreads();
      }
    // Optional SLO floors lo_j <= x_j (max_sum_throughput.py:87-93; L.t carries lo, null = none).  Jobs strictly
    // above the threshold ratio get x = 1, below it their floor; the group TIED at the threshold shares what is left:
    // interior-point selection = max sum 1{lo>0} log(x-lo) + log x + log(1-x) s.t. sum sf x = C over the group
    // (oracle/gavel_lp.py:max_sum_pooled_centre).  One thread finds the group (order-exact sums).
    __shared__ int s_i0, s_i1;
    __shared__ double s_C, s_tot;
    const double *lob = L.t;
    {
      double base = 0.0, bad = 0.0;
      for (int j = threadIdx.x; j < J; j += blockDim.x) {
        const double l = lob ? lob[j] : 0.0;
        if (l > 1.0 + 1e-12) bad += 1.0;
        base += L.sf[j] * l;
      }
      br.sum2(base, bad);
      if (bad > 0.0 || base > N * (1.0 + 1e-12)) status = 1;    // the floors alone do not fit: caller re-solves without them
    }
    if (status == 0) {
    if (threadIdx.x == 0) {
      double used = 0.0, tot = 0.0;
      for (int j = 0; j < J; ++j) { const double l = lob ? fmin(lob[j], 1.0) : 0.0; used += L.sf[j] * l; tot += L.coef[j] * l; }
      int i = 0, g0 = J, g1 = J;
      double C = 0.0;
      while (i < J) {
        const int i0 = i;
        const double r = L.coef[idx[i]] / L.sf[idx[i]];
        double need = 0.0, val = 0.0, floor_w = 0.0;
        while (i < J) {
          const int j = idx[i];
          const double rj = L.coef[j] / L.sf[j];
          if (fabs(rj - r) > 1e-12 * fabs(r)) break;
          const double l = lob ? fmin(lob[j], 1.0) : 0.0;
          need += L.sf[j] * (1.0 - l); val += L.coef[j] * (1.0 - l); floor_w += L.sf[j] * l;
          ++i;
        }
        if (!(r > 0.0)) { g0 = g1 = i0; break; }
        if (used + need <= N) { used += need; tot += val; g0 = g1 = i; }
        else { g0 = i0; g1 = i; C = (N - used) + floor_w; if (!(N - used > 1e-12 * N)) g1 = g0; break; }
      }
      s_i0 = g0; s_i1 = g1; s_C = C; s_tot = tot;
    }
    __syncthreads();
    const int i0 = s_i0, i1 = s_i1;
    const double C = s_C;
    for (int i = threadIdx.x; i < J; i += blockDim.x) {
      const int j = idx[i];
      L.x[j] = i < i0 ? 1.0 : (lob ? fmin(lob[j], 1.0) : 0.0);
    }
    double part = 0.0;
    if (i1 > i0) {
      // x_j(nu): root of 1/x - 1/(1-x) + w/(x-lo) = nu sf on (lo, 1) (decreasing in x and in nu); sum sf x_j(nu) = C
      double xs[POL_MAXJ_PER_THREAD];
      int cnt = 0;
      for (int i = i0 + threadIdx.x; i < i1; i += blockDim.x, ++cnt) {
        const double l = lob ? fmin(lob[idx[i]], 1.0) : 0.0;
        xs[cnt] = 0.5 * (l + 1.0);
      }
      auto load_at = [&](double nu) -> double {
        double load = 0.0;
        int q = 0;
        for (int i = i0 + threadIdx.x; i < i1; i += blockDim.x, ++q) {
          const int j = idx[i];
          const double l0 = lob ? fmin(lob[j], 1.0) : 0.0, w = l0 > 0.0 ? 1.0 : 0.0, ls = nu * L.sf[j];
          double x = xs[q];
          if (l0 >= 1.0) { x = 1.0; }
          else {
            double l = l0, h = 1.0;
            for (int k = 0; k < 80; ++k) {
              const double d1 = 1.0 - x;
              double f = 1.0 / x - 1.0 / d1 - ls, fp = 1.0 / (x * x) + 1.0 / (d1 * d1);
              if (w > 0.0) { const double d0 = x - l0; f += 1.0 / d0; fp += 1.0 / (d0 * d0); }
              if (f == 0.0) break;
              if (f > 0.0) l = x; else h = x;
              double xn = x + f / fp;
              if (xn == x) break;
              if (!(xn > l && xn < h)) xn = 0.5 * (l + h);
              const bool done = fabs(xn - x) <= 2e-15 * xn;
              x = xn;
              if (done) break;
            }
          }
          xs[q] = x;
          load += L.sf[j] * x;
        }
        return br.sum(load);
      };
      // bracket nu by expansion from 0, then bisection (load is decreasing in nu)
      double lo_nu, hi_nu;
      if (load_at(0.0) > C) { lo_nu = 0.0; hi_nu = 1.0; for (int e = 0; e < 60 && load_at(hi_nu) > C; ++e) { lo_nu = hi_nu; hi_nu *= 4.0; } }
      else { hi_nu = 0.0; lo_nu = -1.0; for (int e = 0; e < 60 && load_at(lo_nu) <= C; ++e) { hi_nu = lo_nu; lo_nu *= 4.0; } }
      for (int it = 0; it < 100; ++it) {
        const double nu = 0.5 * (lo_nu + hi_nu);
        if (load_at(nu) > C) lo_nu = nu; else hi_nu = nu;
        if (hi_nu - lo_nu <= 1e-15 * fmax(fabs(hi_nu), fabs(lo_nu))) break;
      }
      load_at(0.5 * (lo_nu + hi_nu));
      int q = 0;
      for (int i = i0 + threadIdx.x; i < i1; i += blockDim.x, ++q) {
        const int j = idx[i];
        const double l = lob ? fmin(lob[j], 1.0) : 0.0;
        L.x[j] = xs[q];
        part += (xs[q] - l) * L.coef[j];
      }
    }
    part = br.sum(part);
    obj = s_tot + part;
    } else {
      for (int j = threadIdx.x; j < J; j += blockDim.x) L.x[j] = 0.0;
    }
  } else if (L.mode == SWB_POL_ISOLATED) {
    // isolated.py:35-55 / proportional.py:26-43 / gandiva_fair_proportional.py:26-41 (pooled):
    // coef_j carries the per-job divisor (sf_j for Isolated, 1 otherwise); rows are normalised to <= 1
    for (int j = threadIdx.x; j < J; j += blockDim.x) {
      const double v = (N / (double)J) / L.coef[j];
      L.x[j] = v > 1.0 ? 1.0 : v;
    }
    obj = 0.0;
  }
  if (threadIdx.x == 0) { L.out[0] = obj; L.out[1] = (double)status; }
}

cudaError_t launch_policy(const PolicyLaunch &L, cudaStream_t st) {
  int npad = 64;
  while (npad < L.J) npad <<= 1;
  size_t smem = 2 * 64 * sizeof(double) + (size_t)npad * (8 + 2) + 64;
  // function attributes are per device: one flag per device ordinal (one process may drive several GPUs)
  static bool attr_done[64] = {false};
  int dev_ = 0;
  cudaGetDevice(&dev_);
  bool &attr_set = attr_done[dev_ & 63];
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(policy_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    if (e != cudaSuccess) return e;
    attr_set = true;
  }
  policy_kernel<<<1, 1024, smem, st>>>(L);
  return cudaGetLastError();
}

}  // namespace swb
