// solve.cu — the per-round market solve of Shockwave on one B200 (sm_100a).
//
// Replaces dynamic_eisenberg_gale_scheduling() (reference scheduler/shockwave.py:504-711): the
// cvxpy model build + Gurobi branch-and-bound.  The MILP's objective depends on x[j][t] only through
// the per-job round counts n_j = sum_t x[j][t] (shockwave.py:371-377), p_j is best at
// min(D n_j / dbar_j, E_j - c_j), and the SOS2 binaries (shockwave.py:403-419) are redundant for a
// concave maximise, so the program collapses to
//     max_n  sum_j w_j plog((c_j + min(D n_j/dbar_j, E_j-c_j))/E_j)/(J T)  -  k max_j rem_j(n_j)
//     s.t.   sum_j g_j n_j <= G T,   nF_j <= n_j <= T            (nF_j from the FTF rows, :573-597)
// which is solved here in its Lagrangian form: a clearing price mu on GPU-rounds found by bisection
// (every job answers a price with a closed-form best response on its piecewise-linear utility)
// nested in a search over the makespan threshold M.  One CTA per scenario.
//
// Hot loop = cost(M, mu) = sum_j g_j n_j(M, mu), evaluated ~10^3 times per solve.  It runs on a
// per-job RESPONSE TABLE staged in shared memory: in the normalised price rho = mu * g_j/(a_j ws_j)
// the thresholds of whole PWL segments are the segment slopes (shared constants), so a job only
// needs, per segment count bs, the number of whole rounds n0[bs] and the threshold ths[bs] of the one
// round that straddles the breakpoint.  ~35 instructions per job and evaluation; reductions are warp
// shuffles + one barrier.  The dense J x T placement of the counts is place.cu.
#include <cooperative_groups.h>
#include <math.h>

#include "swb_common.cuh"
#include "swb_internal.h"

namespace swb {

namespace cg = cooperative_groups;

// Reductions over ALL jobs of a scenario.  CL = 1: the CTA owns every job, plain BlockRed.  CL > 1 (single-scenario
// latency path): a thread-block cluster of CL CTAs splits the jobs; every CTA reduces its slice, publishes the partial
// in its own shared memory and, after one cluster barrier, every thread of every CTA adds up the CL partials through
// distributed shared memory IN RANK ORDER — all CTAs see bit-identical totals, so the (data-dependent) control flow
// of the price / makespan searches stays uniform across the cluster.  Two slots used alternately: a CTA that races
// ahead into reduction k+1 writes the other slot and cannot reach k+2 before everyone has left k's barrier.
template <int CL>
struct ClusterRed {
  BlockRed br;
  double *xs;        // this CTA's published partials: [2 slots][2 values]
  int *xw;           // [2 slots][32 warps][3]: per-WARP partials of sumi3, read by every CTA of the cluster
  int xphase, wphase;
  __device__ __forceinline__ ClusterRed(double *scratch, double *xslots)
      : br(scratch), xs(xslots), xw(reinterpret_cast<int *>(xslots + 4)), xphase(0), wphase(0) {}

  __device__ __forceinline__ void exchange2(double &a, double &b, int op) {   // op 0: sum, 1: max
    if constexpr (CL > 1) {
      cg::cluster_group cl = cg::this_cluster();
      if (threadIdx.x == 0) { xs[xphase * 2] = a; xs[xphase * 2 + 1] = b; }
      cl.sync();
      double ra = op ? -1.0e300 : 0.0, rb = 0.0;
#pragma unroll
      for (int r = 0; r < CL; ++r) {
        const double *rem = cl.map_shared_rank(xs, r);
        const double va = rem[xphase * 2], vb = rem[xphase * 2 + 1];
        if (op) ra = fmax(ra, va); else { ra += va; rb += vb; }
      }
      a = ra; b = rb;
      xphase ^= 1;
    }
  }
  __device__ __forceinline__ void sum2(double &a, double &b) { br.sum2(a, b); exchange2(a, b, 0); }
  __device__ __forceinline__ double sum(double a) { double b = 0.0; sum2(a, b); return a; }
  __device__ __forceinline__ long long sumll(long long a) {
    a = br.sumll(a);
    if constexpr (CL > 1) {
      // exact in a double pair: hi = a / 2^26, lo = a mod 2^26 (|a| < 2^52 here: GPU-rounds, counts)
      double hi = (double)(a >> 26), lo = (double)(a & ((1ll << 26) - 1));
      exchange2(hi, lo, 0);
      a = ((long long)hi << 26) + (long long)lo;
    }
    return a;
  }
  // demand sums: int32 (J * 255 * T < 2^31), REDUX inside the CTA, one 32-bit slot per CTA across the cluster
  __device__ __forceinline__ int sumi(int a) {
    a = br.sumi(a);
    if constexpr (CL > 1) {
      cg::cluster_group cl = cg::this_cluster();
      int *xi = reinterpret_cast<int *>(xs);
      if (threadIdx.x == 0) xi[xphase * 4] = a;
      cl.sync();
      int r = 0;
#pragma unroll
      for (int q = 0; q < CL; ++q) r += reinterpret_cast<const int *>(cl.map_shared_rank(xs, q))[xphase * 4];
      a = r;
      xphase ^= 1;
    }
    return a;
  }
  // three demand sums per pass: block reduction first, then ONE 16-byte slot per CTA through distributed shared memory.
  // (Publishing the per-warp partials instead and letting the cluster barrier double as the block barrier was measured
  // twice as slow: 16 lanes x 8 CTAs x 3 remote loads per warp saturate the ~17 B/clk DSMEM port.)
  __device__ __forceinline__ void sumi3(int &a, int &b, int &c) {
    br.sumi3(a, b, c);
    if constexpr (CL > 1) {
      cg::cluster_group cl = cg::this_cluster();
      int *xi = reinterpret_cast<int *>(xs);                    // a slot is 16 bytes: three ints fit
      if (threadIdx.x == 0) { xi[xphase * 4] = a; xi[xphase * 4 + 1] = b; xi[xphase * 4 + 2] = c; }
      cl.sync();
      int ra = 0, rb = 0, rc = 0;
#pragma unroll
      for (int q = 0; q < CL; ++q) {
        const int *rem = reinterpret_cast<const int *>(cl.map_shared_rank(xs, q)) + xphase * 4;
        ra += rem[0]; rb += rem[1]; rc += rem[2];
      }
      a = ra; b = rb; c = rc;
      xphase ^= 1;
    }
  }
  __device__ __forceinline__ double max(double a) { a = br.max(a); double b = 0.0; exchange2(a, b, 1); return a; }
  __device__ __forceinline__ double min(double a) { return -max(-a); }
  // all-gather of one value per CTA (rank order) — used for the prefix of the tie-fill
  __device__ __forceinline__ long long prefix_of_rank(long long mine, int rank) {
    if constexpr (CL > 1) {
      cg::cluster_group cl = cg::this_cluster();
      if (threadIdx.x == 0) { xs[xphase * 2] = (double)mine; xs[xphase * 2 + 1] = 0.0; }
      cl.sync();
      long long pre = 0;
      for (int r = 0; r < rank; ++r) pre += (long long)cl.map_shared_rank(xs, r)[xphase * 2];
      xphase ^= 1;
      return pre;
    } else {
      return 0;
    }
  }
};

struct Tab {             // response table: shared memory for J <= SWB_SMEM_JOBS, else global scratch
  double *cth, *R;       // rho = mu * cth ; remaining runtime IN ROUNDS (R_j / D)
  float *ths;            // [J][B] straddle-round threshold in rho units (-1: no such round)
  uint8_t *n0;           // [J][B] whole rounds inside the segments whose slope beats rho
  uint8_t *g, *nF, *nmax;
};

struct Ctx {
  const Pwl *P;
  Tab t;
  float sl[8];           // PWL segment slopes as float registers (B <= 9), padded with -inf
  const double *Rsec;    // remaining runtime in seconds (global scratch) for the exact makespan passes
  // exact per-job constants, global scratch (read ~20x per solve: welfare / makespan passes)
  double *a, *u0, *ws, *cap;
  uint8_t *n;
  int J, T, GT, B;
  int j0, j1;           // this CTA's slice of the jobs ([0, J) unless the scenario is split over a cluster)
  double D, invD;
};

// best response of job j to the price mu: the largest n with F_j(n) - F_j(n-1) > mu g_j.
// The normalised price is compared in fp32 (thresholds are O(1..60) slopes); every caller goes through
// this one function, so the step function it defines is consistent (monotone in mu) everywhere.
__device__ __forceinline__ int pref_n(const Ctx &c, int j, double mu) {
  if (mu <= 0.0) return c.t.nmax[j];
  const float rho = __double2float_rn(mu * c.t.cth[j]);
  int bs = 0;
#pragma unroll
  for (int b = 0; b < 8; ++b) bs += (c.sl[b] > rho) ? 1 : 0;
  const int i = j * c.B + bs;
  return (int)c.t.n0[i] + ((rho < c.t.ths[i]) ? 1 : 0);
}

// rounds job j must get so that rem_j <= M  (rem_j = max(0, R_j - min(D n, cap_j))); Md = M / D
__device__ __forceinline__ int lower_n(const Ctx &c, int j, double Md) {
  const double need = c.t.R[j] - Md;
  int L = 0;
  if (need > 0.0) L = min((int)c.t.nmax[j], __double2int_ru(need - 1e-9));
  return max(L, (int)c.t.nF[j]);
}

__device__ __forceinline__ int job_n(const Ctx &c, int j, double Md, double mu) {
  return max(lower_n(c, j, Md), pref_n(c, j, mu));
}

__device__ __forceinline__ double rem_of(const Ctx &c, int j, int n) {
  const double done = fmin(c.D * (double)n, c.cap[j]);
  return fmax(0.0, c.Rsec[j] - done);
}

// weighted PWL-log utility of n rounds
__device__ __forceinline__ double util_of(const Ctx &c, int j, int n) {
  const double u = util_u(c.a[j], c.u0[j], c.cap[j], c.D, n);
  return c.ws[j] * plog(*c.P, u);
}

template <class Red>
__device__ long long cost_at(const Ctx &c, Red &br, double M, double mu) {
  const double Md = M * c.invD;
  int s = 0;
#pragma unroll 4
  for (int j = c.j0 + threadIdx.x; j < c.j1; j += blockDim.x) s += (int)c.t.g[j] * job_n(c, j, Md, mu);
  return (long long)br.sumi(s);
}

// demand at three prices in one pass over the jobs and ONE reduction: an evaluation costs a block (cluster) barrier,
// not arithmetic, so three candidates per barrier shorten the search by the number of passes it saves
template <class Red>
__device__ void cost_at3(const Ctx &c, Red &br, double M, double mu0, double mu1, double mu2, long long &c0,
                         long long &c1, long long &c2) {
  const double Md = M * c.invD;
  int s0 = 0, s1 = 0, s2 = 0;
#pragma unroll 2
  for (int j = c.j0 + threadIdx.x; j < c.j1; j += blockDim.x) {
    const int L = lower_n(c, j, Md), g = (int)c.t.g[j];
    s0 += g * max(L, pref_n(c, j, mu0));
    s1 += g * max(L, pref_n(c, j, mu1));
    s2 += g * max(L, pref_n(c, j, mu2));
  }
  br.sumi3(s0, s1, s2);
  c0 = s0; c1 = s1; c2 = s2;
}

struct Price { double hi, lo; long long cost_hi; int iters; };

// smallest price at which demand fits: cost(M, hi) <= GT < cost(M, lo).
// Search on the BIT PATTERN of the (positive) price: the fallback priorities span 20+ orders of
// magnitude (ratio^lam, shockwave.py:899-903), so an arithmetic midpoint would stop far above the real
// clearing price and lump every cheaper item into one "tie".  Positive doubles are ordered like their bit
// patterns.  The loop ends when hi/lo - 1 < 2^-prec; everything priced inside such an interval is treated
// as a tie and filled in job order (prec = 12 while searching the makespan threshold, 22 for the final
// allocation; the response function itself has fp32 resolution).  `hint` (> 0) is the clearing price of a
// neighbouring threshold: the search then starts from [hint/4, 4 hint] when that bracket holds.
// Every pass evaluates THREE prices (cost_at3): the first one the free price 0 and both ends of the hint bracket, the
// later ones the regula-falsi point of the bracket (the excess demand is a step function, but close to linear in
// log(price) at the scale of the bracket) flanked at +-1/8 of the bracket; a pass that shrinks the bracket by less
// than half is followed by a pass at the quarter points (guaranteed factor 4), so the worst case stays logarithmic.
template <class Red>
__device__ Price solve_price(const Ctx &c, Red &br, double M, double mu_max, int prec, double hint) {
  Price p;
  p.iters = 1;
  const double h4 = hint > 0.0 ? fmin(mu_max, hint * 4.0) : mu_max, l4 = hint > 0.0 ? hint * 0.25 : mu_max;
  long long c0, ch, cl;
  cost_at3(c, br, M, 0.0, h4, l4, c0, ch, cl);
  if (c0 <= c.GT) { p.hi = p.lo = 0.0; p.cost_hi = c0; return p; }
  unsigned long long lob = 0ull, hib = (unsigned long long)__double_as_longlong(mu_max);
  double lo = 0.0, hi = mu_max;
  long long chi = -1, clo = -1;     // demand at hi / at lo (-1: not evaluated; lo = 0 has no log-scale position)
  if (hint > 0.0) {
    if (ch <= c.GT) { hi = h4; hib = (unsigned long long)__double_as_longlong(h4); chi = ch; }
    if (cl > c.GT) { lo = l4; lob = (unsigned long long)__double_as_longlong(l4); clo = cl; }
    else if (chi >= 0 || l4 < hi) { hi = l4; hib = (unsigned long long)__double_as_longlong(l4); chi = cl; }
  } else {
    chi = ch;                       // h4 = mu_max
  }
  if (chi < 0) { chi = cost_at(c, br, M, hi); p.iters++; }
  const unsigned long long width = 1ull << (52 - prec);
  double flo = clo >= 0 ? (double)(clo - c.GT) : -1.0, fhi = (double)(chi - c.GT);
  bool quarters = false;
  while (hib - lob > width && fhi != 0.0) {
    const unsigned long long span = hib - lob;
    double f1 = 0.25, f2 = 0.5, f3 = 0.75;
    if (!quarters && flo > 0.0 && fhi < 0.0 && lob != 0ull) {
      f2 = fmin(0.85, fmax(0.15, flo / (flo - fhi)));
      f1 = f2 - 0.125; f3 = f2 + 0.125;
    }
    unsigned long long b1 = lob + (unsigned long long)((double)span * f1);
    unsigned long long b2 = lob + (unsigned long long)((double)span * f2);
    unsigned long long b3 = lob + (unsigned long long)((double)span * f3);
    if (b1 <= lob) b1 = lob + 1;
    if (b2 <= b1) b2 = b1 + 1;
    if (b3 <= b2) b3 = b2 + 1;
    if (b3 >= hib) b3 = hib - 1;              // span > width >= 2^30: the three points stay distinct and interior
    const double m1 = __longlong_as_double((long long)b1), m2 = __longlong_as_double((long long)b2),
                 m3 = __longlong_as_double((long long)b3);
    long long k1, k2, k3;
    cost_at3(c, br, M, m1, m2, m3, k1, k2, k3);
    p.iters++;
    // demand is non-increasing in the price: the new bracket is the sub-interval where it crosses GT
    if (k1 <= c.GT) { hib = b1; hi = m1; chi = k1; }
    else if (k2 <= c.GT) { lob = b1; lo = m1; clo = k1; hib = b2; hi = m2; chi = k2; }
    else if (k3 <= c.GT) { lob = b2; lo = m2; clo = k2; hib = b3; hi = m3; chi = k3; }
    else { lob = b3; lo = m3; clo = k3; }
    flo = clo >= 0 ? (double)(clo - c.GT) : -1.0;
    fhi = (double)(chi - c.GT);
    quarters = (hib - lob) > (span >> 1);
  }
  p.hi = hi; p.lo = lo; p.cost_hi = chi;
  return p;
}

struct Phi { double V, welfare, Meff, mu; long long cost; };

// value of makespan threshold M: LP-style welfare at the clearing price minus k * achieved makespan
template <class Red>
__device__ Phi phi_at(const Ctx &c, Red &br, double M, double mu_max, double k, int &iters, double hint) {
  Price p = solve_price(c, br, M, mu_max, 12, hint);
  iters += p.iters;
  double w = 0.0, me = 0.0;
  const double Md = M * c.invD;
  for (int j = c.j0 + threadIdx.x; j < c.j1; j += blockDim.x) {
    const int n = job_n(c, j, Md, p.hi);
    w += util_of(c, j, n);
    me = fmax(me, rem_of(c, j, n));
  }
  w = br.sum(w);
  me = br.max(me);
  Phi r;
  r.welfare = w; r.Meff = me; r.mu = p.hi; r.cost = p.cost_hi;
  r.V = w + p.hi * (double)(c.GT - p.cost_hi) - k * me;
  return r;
}

// ---- exact optimum of the CONTINUOUS relaxation (x in [0,1], hence n_j real): parity item P4 ----------
// Same Lagrangian structure with real-valued responses: a job's best n is a breakpoint of its PWL utility,
// ties at the clearing price absorb the left-over capacity fractionally (their utility is linear there),
// and the value is concave in the makespan threshold, so a golden-section search is exact.
struct RelaxCtx { const double *nfc; double Tr; };

__device__ __forceinline__ double nmax_real(const Ctx &c, const RelaxCtx &r, int j) {
  return c.t.nmax[j] == 0 ? 0.0 : fmin(r.Tr, fmin(c.cap[j] * c.invD, (double)c.t.nmax[j]));
}

__device__ __forceinline__ double job_nc(const Ctx &c, const RelaxCtx &r, int j, double Md, double mu) {
  const double nm = nmax_real(c, r, j);
  double lb = fmax(r.nfc[j], fmax(0.0, c.t.R[j] - Md));
  lb = fmin(lb, nm);
  double pf = nm;
  if (mu > 0.0) {
    const float rho = __double2float_rn(mu * c.t.cth[j]);
    int bs = 0;
#pragma unroll
    for (int b = 0; b < 8; ++b) bs += (c.sl[b] > rho) ? 1 : 0;
    pf = bs == 0 ? 0.0 : fmin(nm, fmax(0.0, (c.P->base[bs] - c.u0[j]) / c.a[j]));
  }
  return fmax(lb, pf);
}

__device__ __forceinline__ double util_c(const Ctx &c, int j, double n) {
  const double u = (c.D * n >= c.cap[j]) ? 1.0 : fma(c.a[j], n, c.u0[j]);
  return c.ws[j] * plog(*c.P, u);
}

template <class Red>
__device__ double cost_c(const Ctx &c, const RelaxCtx &r, Red &br, double Md, double mu) {
  double s = 0.0;
  for (int j = c.j0 + threadIdx.x; j < c.j1; j += blockDim.x) s += (double)c.t.g[j] * job_nc(c, r, j, Md, mu);
  return br.sum(s);
}

template <class Red>
__device__ double phi_c(const Ctx &c, const RelaxCtx &r, Red &br, double M, double mu_max, double k) {
  const double Md = M * c.invD, cap = (double)c.GT;
  double mu = 0.0, c_hi = cost_c(c, r, br, Md, 0.0), c_lo = c_hi;
  if (c_hi > cap * (1.0 + 1e-13)) {
    unsigned long long lob = 0ull, hib = (unsigned long long)__double_as_longlong(mu_max);
    c_lo = c_hi;
    c_hi = cost_c(c, r, br, Md, mu_max);
    mu = mu_max;
    while (hib - lob > (1ull << 20)) {
      const unsigned long long midb = lob + ((hib - lob) >> 1);
      const double mid = __longlong_as_double((long long)midb);
      const double cm = cost_c(c, r, br, Md, mid);
      if (cm <= cap * (1.0 + 1e-13)) { hib = midb; mu = mid; c_hi = cm; } else { lob = midb; c_lo = cm; }
    }
  }
  double w = 0.0, me = 0.0;
  for (int j = c.j0 + threadIdx.x; j < c.j1; j += blockDim.x) {
    const double n = job_nc(c, r, j, Md, mu);
    w += util_c(c, j, n);
    me = fmax(me, fmax(0.0, c.Rsec[j] - fmin(c.D * n, c.cap[j])));
  }
  w = br.sum(w);
  me = br.max(me);
  const double fill = fmax(0.0, fmin(cap - c_hi, c_lo - c_hi));   // tied jobs take the rest, utility linear
  return w + mu * fill - k * me;
}

template <class Red>
__device__ double relaxed_optimum(const Ctx &c, const RelaxCtx &r, Red &br, double mu_max, double k) {
  // makespan threshold range: floor (everybody at its continuous maximum) .. natural (no threshold)
  double mfl = 0.0, mtop = 0.0;
  for (int j = c.j0 + threadIdx.x; j < c.j1; j += blockDim.x) {
    const double nm = nmax_real(c, r, j);
    mfl = fmax(mfl, c.Rsec[j] - fmin(c.D * nm, c.cap[j]));
    mtop = fmax(mtop, c.Rsec[j]);
  }
  mfl = fmax(0.0, br.max(mfl));
  mtop = br.max(mtop);
  // smallest threshold whose forced demand fits
  double lo = mfl, hi = mtop;
  if (cost_c(c, r, br, mfl * c.invD, mu_max) > (double)c.GT) {
    for (int it = 0; it < 80; ++it) {
      const double mid = 0.5 * (lo + hi);
      if (cost_c(c, r, br, mid * c.invD, mu_max) <= (double)c.GT) hi = mid; else lo = mid;
    }
    lo = hi;
  }
  hi = mtop;
  double best = fmax(phi_c(c, r, br, lo, mu_max, k), phi_c(c, r, br, hi, mu_max, k));
  const double gr = 0.6180339887498949;
  double x1 = hi - gr * (hi - lo), x2 = lo + gr * (hi - lo);
  double f1 = phi_c(c, r, br, x1, mu_max, k), f2 = phi_c(c, r, br, x2, mu_max, k);
  for (int it = 0; it < 70 && hi - lo > 1e-9 * (1.0 + hi); ++it) {
    if (f1 < f2) { lo = x1; x1 = x2; f1 = f2; x2 = lo + gr * (hi - lo); f2 = phi_c(c, r, br, x2, mu_max, k); }
    else { hi = x2; x2 = x1; f2 = f1; x1 = hi - gr * (hi - lo); f1 = phi_c(c, r, br, x1, mu_max, k); }
    best = fmax(best, fmax(f1, f2));
  }
  return best;
}

// SMEM = the response table lives in shared memory (J <= SWB_SMEM_JOBS).  A compile-time switch so that
// the hot loop's accesses are LDS with 32-bit addresses instead of generic 64-bit loads.
template <bool SMEM, int NT, int CL>
__global__ void __launch_bounds__(NT, 1) solve_kernel(SolveLaunch L) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int s = blockIdx.x / CL;
  int rank = 0;
  if constexpr (CL > 1) rank = (int)cg::this_cluster().block_rank();
  const int J = L.J;
  // this CTA's slice of the jobs (whole warps, so that the slices of a cluster are contiguous in job order)
  const int Jc = CL > 1 ? ((((J + CL - 1) / CL) + 31) & ~31) : J;
  const int jbeg = rank * Jc < J ? rank * Jc : J, jend = (jbeg + Jc < J) ? jbeg + Jc : J;
  const swb_params &prm = L.prm[s];
  const int T = prm.future_rounds, G = prm.ngpus, B = prm.nbases;
  const double D = prm.round_duration, k = prm.k;

  // ---- shared-memory carve-up -------------------------------------------------------------
  Pwl *P = reinterpret_cast<Pwl *>(smem_raw);
  double *red = reinterpret_cast<double *>(smem_raw + SWB_PWL_BYTES);  // 2*64 doubles
  double *xslots = red + 2 * 64;                                       // 4 doubles: cluster exchange slots
  unsigned char *p = smem_raw + SWB_PWL_BYTES + (2 * 64 + 4) * sizeof(double) + 2 * 96 * sizeof(int);   // + xw
  Ctx c;
  c.j0 = jbeg; c.j1 = jend;
  const size_t so = (size_t)s * J;
  if constexpr (SMEM) {
    // the table holds this CTA's Jc jobs; the pointers are shifted so that the GLOBAL job index addresses it
    c.t.cth = reinterpret_cast<double *>(p) - jbeg; p += sizeof(double) * Jc;
    c.t.R = reinterpret_cast<double *>(p) - jbeg;   p += sizeof(double) * Jc;
    c.t.ths = reinterpret_cast<float *>(p) - (size_t)jbeg * B;  p += sizeof(float) * Jc * B;
    c.t.n0 = p - (size_t)jbeg * B;   p += (size_t)Jc * B;
    c.t.g = p - jbeg;    p += Jc;
    c.t.nF = p - jbeg;   p += Jc;
    c.t.nmax = p - jbeg; p += Jc;
  } else {
    c.t.cth = L.sc_cth + so; c.t.R = L.sc_Rr + so;
    c.t.ths = L.sc_ths + so * SWB_MAX_BASES; c.t.n0 = L.sc_n0 + so * SWB_MAX_BASES;
    c.t.g = L.sc_g + so; c.t.nF = L.sc_nF + so; c.t.nmax = L.sc_nmax + so;
  }
  c.a = L.sc_a + so; c.u0 = L.sc_u0 + so; c.ws = L.sc_ws + so; c.cap = L.sc_cap + so;
  c.n = L.sc_n + so;
  c.P = P; c.J = J; c.T = T; c.GT = G * T; c.B = B; c.D = D; c.invD = 1.0 / D;
  c.Rsec = L.sc_R + so;
  ClusterRed<CL> br(red, xslots);
#pragma unroll
  for (int b = 0; b < 8; ++b)
    c.sl[b] = (b + 1 < B) ? (float)((prm.logv[b + 1] - prm.logv[b]) / (prm.bases[b + 1] - prm.bases[b])) : -INFINITY;

  if (threadIdx.x == 0) make_pwl(*P, prm);
  __syncthreads();

  const size_t jo = L.per_scn ? so : 0;
  const int32_t *gI = L.g + jo, *EI = L.E + jo, *cI = L.c + jo;
  const double *dbarI = L.dbar + jo, *RI = L.rem + jo, *ftI = L.ftobj + jo;
  const double *RfbI = L.rem_fb ? L.rem_fb + jo : RI;
  const double share = fmin(1.0, (double)G / (double)J);
  const double invJT = 1.0 / ((double)J * (double)T);
  const double next_t = D * (double)(prm.round_ptr + T);

  // ---- phase 1: job constants + finish-time-fairness rows (shockwave.py:573-597) -----------
  long long infeasible = 0, forced = 0;
  int badw = 0;      // gang widths are bytes from here on: anything outside [1,255] is reported, never truncated
  for (int j = c.j0 + threadIdx.x; j < c.j1; j += blockDim.x) {
    const double Ef = (double)EI[j], cf = (double)cI[j], dbar = dbarI[j], R = RI[j];
    const double cap = dbar * (Ef - cf);
    const double a = D / (dbar * Ef);
    int nfin = cap <= 0.0 ? 0 : (int)fmin(ceil(cap / D - 1e-9), 255.0);
    int nmax = nfin < T ? nfin : T;
    const int gw = gI[j];
    if (gw < 1 || gw > 255) { badw = 1; nmax = 0; }
    if (gw > G) nmax = 0;  // a gang wider than the cluster violates every capacity row (shockwave.py:317)
    if (L.ncap && (int)L.ncap[so + j] < nmax) nmax = L.ncap[so + j];  // packing feedback (written by place_kernel)
    c.a[j] = a; c.u0[j] = cf / Ef; c.cap[j] = cap;
    c.t.R[j] = R * c.invD; L.sc_R[so + j] = R;   // rounds (table) and seconds (exact passes): distinct buffers
    c.t.g[j] = (uint8_t)(gw < 1 ? 1 : (gw > 255 ? 255 : gw)); c.t.nmax[j] = (uint8_t)nmax;
    const double capF = share * (prm.rhomax * ftI[j] - next_t);
    int nF = 0, bad = 0;
    if (capF < 0.0) bad = 1;
    else {
      const double need = R - capF;
      if (need > 0.0) {
        if (need > cap * (1.0 + 1e-12) + 1e-9) bad = 1;
        else {
          const double q = ceil(need / D - 1e-9);
          // q > nmax with q <= T: either the packing feedback capped the job (ncap: keep the plan, seat what fits)
          // or the gang is wider than the cluster — then the reference's row shockwave.py:586-590 cannot hold with
          // x_j = 0 and its MILP is infeasible -> fallback verdict
          if (q > (double)nmax) { if (q > (double)T || gw > G) bad = 1; else nF = nmax; }
          else nF = (int)q;
        }
      }
    }
    c.t.nF[j] = (uint8_t)nF;
    if (L.sc_nfc) L.sc_nfc[so + j] = (!bad && R - capF > 0.0) ? (R - capF) / D : 0.0;
    infeasible += bad;
    forced += (long long)gw * nF;
  }
  infeasible = br.sumll(infeasible);
  forced = br.sumll(forced);
  badw = (int)br.sumll((long long)badw);
  const bool ftf_ok = (infeasible == 0) && (forced <= (long long)c.GT);

  // fallback priorities (shockwave.py:830-911); weights stay 1 when the FTF rows are satisfiable.
  // Then the response table of the job (see the file header).
  double mu_max = 0.0, mfloor = 0.0, mtop = 0.0;
  for (int j = c.j0 + threadIdx.x; j < c.j1; j += blockDim.x) {
    double w = 1.0;
    if (!ftf_ok) {
      c.t.nF[j] = 0;
      if (L.sc_nfc) L.sc_nfc[so + j] = 0.0;
      const double R = RfbI[j];
      const double ratio = (D * (double)prm.round_ptr + R / share) / ftI[j];
      if (ratio > prm.rhomax) {
        w = pow(ratio, (R < D) ? 1e2 : prm.lam);
        w = fmin(w, 1e300);
      }
    }
    const double ws = w * invJT;
    c.ws[j] = ws;
    if (L.weights) L.weights[so + j] = w;
    const double a = c.a[j], u0 = c.u0[j], cap = c.cap[j];
    const int nmax = c.t.nmax[j];
    c.t.cth[j] = (double)c.t.g[j] / (a * ws);
    for (int bs = 0; bs < B; ++bs) {
      int n0 = 0;
      if (bs > 0) {
        const double nb = (P->base[bs] - u0) / a;
        n0 = nb <= 0.0 ? 0 : (nb >= (double)nmax ? nmax : (int)floor(nb));
      }
      float th = -1.0f;
      if (n0 < nmax) {
        const double u1 = util_u(a, u0, cap, D, n0 + 1), u_0 = util_u(a, u0, cap, D, n0);
        th = (float)((plog(*P, u1) - plog(*P, u_0)) / a);
      }
      c.t.n0[j * B + bs] = (uint8_t)n0;
      c.t.ths[j * B + bs] = th;
    }
    if (nmax > 0) mu_max = fmax(mu_max, (util_of(c, j, 1) - util_of(c, j, 0)) / (double)c.t.g[j]);
    const double R = c.Rsec[j];
    mfloor = fmax(mfloor, R - fmin(D * (double)nmax, cap));
    mtop = fmax(mtop, R);
  }
  // ---- phase 2: price ceiling, makespan floor, smallest packable makespan -------------------
  mu_max = br.max(mu_max) * (1.0 + 1e-6) + 1e-300;
  mfloor = fmax(0.0, br.max(mfloor));
  mtop = br.max(mtop);
  __syncthreads();
  const double INF_M = 1e300;
  const double eps = 1e-6 * D;

  int m_evals = 0, iters = 0;
  double mmin = mfloor;
  if (cost_at(c, br, mfloor, mu_max) > c.GT) {  // forced demand only at the price ceiling
    double lo = mfloor, hi = mtop;
    for (int it = 0; it < 60 && hi - lo > 1e-9 * (1.0 + hi); ++it) {
      const double mid = 0.5 * (lo + hi);
      if (cost_at(c, br, mid, mu_max) <= c.GT) hi = mid; else lo = mid;
      iters++;
    }
    mmin = hi;
  }

  // ---- phase 3: search the makespan threshold (value is concave in the relaxation) ----------
  Phi nat = phi_at(c, br, INF_M, mu_max, k, iters, 0.0); m_evals++;
  double hint = nat.mu;
  double best_V = nat.V, best_thr = INF_M;
  if (nat.Meff - eps >= mmin) {
    Phi t2 = phi_at(c, br, nat.Meff - eps, mu_max, k, iters, hint); m_evals++;
    if (t2.V > nat.V) {
      best_V = t2.V; best_thr = nat.Meff - eps;
      double lo = mmin, hi = nat.Meff - eps;
      Phi pl = phi_at(c, br, lo, mu_max, k, iters, hint); m_evals++;
      if (pl.V > best_V) { best_V = pl.V; best_thr = lo; }
      for (int it = 0; it < 48 && hi - lo > eps; ++it) {
        const double mid = 0.5 * (lo + hi);
        Phi p1 = phi_at(c, br, mid, mu_max, k, iters, hint); m_evals++;
        if (p1.mu > 0.0) hint = p1.mu;
        if (p1.V > best_V) { best_V = p1.V; best_thr = mid; }
        const double below = p1.Meff - eps;
        if (below < mmin) break;               // already at the smallest packable makespan
        Phi p2 = phi_at(c, br, below, mu_max, k, iters, p1.mu > 0.0 ? p1.mu : hint); m_evals++;
        if (p2.V > best_V) { best_V = p2.V; best_thr = below; }
        if (p2.V > p1.V) hi = below; else lo = mid;
      }
    }
  }

  // ---- phase 4: integral allocation at the chosen threshold ----------------------------------
  Price pr = solve_price(c, br, best_thr, mu_max, 22, hint);
  iters += pr.iters;
  const double thr_d = best_thr * c.invD;
  for (int j = c.j0 + threadIdx.x; j < c.j1; j += blockDim.x) c.n[j] = (uint8_t)job_n(c, j, thr_d, pr.hi);
  long long left = (long long)c.GT - pr.cost_hi;
  __syncthreads();

  // (a) ties at the clearing price: jobs whose demand jumps between pr.lo and pr.hi, in job order
  //     (cluster: the carry into this CTA's slice is the tie demand of the lower ranks)
  __shared__ long long s_carry;
  __shared__ long long s_wsum[32];
  if (left > 0 && pr.lo < pr.hi) {
    long long mine = 0;
    if constexpr (CL > 1) {
      for (int j = c.j0 + threadIdx.x; j < c.j1; j += blockDim.x) {
        int extra = job_n(c, j, thr_d, pr.lo) - (int)c.n[j];
        if (extra > 0) mine += (long long)c.t.g[j] * extra;
      }
      mine = br.br.sumll(mine);
    }
    const long long carry0 = br.prefix_of_rank(mine, rank);
    if (threadIdx.x == 0) s_carry = carry0;
    __syncthreads();
    for (int base = c.j0; base < c.j1; base += blockDim.x) {
      const int j = base + threadIdx.x;
      int extra = 0, gj = 1;
      if (j < c.j1) { gj = c.t.g[j]; extra = job_n(c, j, thr_d, pr.lo) - (int)c.n[j]; if (extra < 0) extra = 0; }
      long long v = (long long)gj * extra, incl = v;
      for (int o = 1; o < 32; o <<= 1) {
        long long t = __shfl_up_sync(SWB_FULL, incl, o);
        if ((threadIdx.x & 31) >= o) incl += t;
      }
      if ((threadIdx.x & 31) == 31) s_wsum[threadIdx.x >> 5] = incl;
      __syncthreads();
      long long woff = 0;
      for (int w = 0; w < (int)(threadIdx.x >> 5); ++w) woff += s_wsum[w];
      const long long carry = s_carry;
      const long long excl = carry + woff + incl - v;
      if (j < c.j1 && extra > 0) {
        long long room = left - excl;
        if (room > 0) {
          long long take = room / gj;
          if (take > extra) take = extra;
          c.n[j] = (uint8_t)(c.n[j] + take);
        }
      }
      __syncthreads();
      if (threadIdx.x == blockDim.x - 1) s_carry = carry + woff + incl;
      __syncthreads();
    }
  }
  __syncthreads();
  // (b) completion: best remaining item that still fits, a few times
  {
    long long used = 0;
    for (int j = c.j0 + threadIdx.x; j < c.j1; j += blockDim.x) used += (long long)c.t.g[j] * c.n[j];
    used = br.sumll(used);
    left = (long long)c.GT - used;
    for (int rep = 0; rep < 32 && left > 0; ++rep) {
      double bd = 0.0;
      for (int j = c.j0 + threadIdx.x; j < c.j1; j += blockDim.x) {
        const int n = c.n[j];
        if (n < c.t.nmax[j] && (long long)c.t.g[j] <= left)
          bd = fmax(bd, (util_of(c, j, n + 1) - util_of(c, j, n)) / (double)c.t.g[j]);
      }
      bd = br.max(bd);
      if (!(bd > 0.0)) break;
      double bj = 1e300;
      for (int j = c.j0 + threadIdx.x; j < c.j1; j += blockDim.x) {
        const int n = c.n[j];
        if (n < c.t.nmax[j] && (long long)c.t.g[j] <= left &&
            (util_of(c, j, n + 1) - util_of(c, j, n)) / (double)c.t.g[j] >= bd)
          bj = fmin(bj, (double)j);
      }
      bj = br.min(bj);
      if (bj >= 1e299) break;
      const int wj = (int)bj;
      // the CTA that owns job wj applies the step; its width reaches the others through a cluster reduction
      double gw = 0.0;
      if (wj >= c.j0 && wj < c.j1) {
        if (threadIdx.x == 0) { c.n[wj] = (uint8_t)(c.n[wj] + 1); gw = (double)c.t.g[wj]; }
      }
      if constexpr (CL > 1) gw = br.max(gw); else gw = (double)c.t.g[wj];
      left -= (long long)gw;
      __syncthreads();
    }
  }

  // ---- phase 5: scalars of the plan; constants the placement kernel re-reads ------------------
  double w = 0.0, me = 0.0;
  for (int j = c.j0 + threadIdx.x; j < c.j1; j += blockDim.x) {
    const int n = c.n[j];
    w += util_of(c, j, n);
    me = fmax(me, rem_of(c, j, n));
    if constexpr (SMEM) { L.sc_g[so + j] = c.t.g[j]; L.sc_nF[so + j] = c.t.nF[j]; L.sc_nmax[so + j] = c.t.nmax[j]; }
  }
  w = br.sum(w);
  me = br.max(me);
  if (threadIdx.x == 0 && rank == 0) {
    swb_result &r = L.res[s];
    r.status = ftf_ok ? SWB_ST_OK : SWB_ST_FALLBACK;
    r.m_evals = m_evals;
    r.mu_iters = iters;
    r.shortfall = 0;
    r.flags = badw ? 1 : 0;
    r.welfare = w;
    r.makespan = me;
    r.objective = w - k * me;
    r.price = pr.hi;
    r.relaxed_objective = best_V;
  }
  if (L.want_relaxed && L.sc_nfc) {
    __syncthreads();
    RelaxCtx rc;
    rc.nfc = L.sc_nfc + so; rc.Tr = (double)T;
    const double rv = relaxed_optimum(c, rc, br, mu_max, k);
    if (threadIdx.x == 0 && rank == 0) L.res[s].relaxed_objective = rv;
  }
  if constexpr (CL > 1) cg::this_cluster().sync();   // nobody leaves while its exchange slots may still be read
}

template <class K>
static cudaError_t set_smem_attr(K kern, int static_bytes) {
  return cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SWB_MAX_DYN_SMEM - static_bytes);
}

cudaError_t launch_solve(const SolveLaunch &L, cudaStream_t st, int nbases) {
  const size_t smem_fixed = SWB_PWL_BYTES + (2 * 64 + 4) * sizeof(double) + 2 * 96 * sizeof(int);
  // function attributes are per device: one flag per device ordinal (one process may drive several GPUs)
  static bool attr_done[64] = {false};
  int dev_ = 0;
  cudaGetDevice(&dev_);
  bool &attr_set = attr_done[dev_ & 63];
  if (!attr_set) {
    cudaFuncAttributes fa;
    cudaError_t e = cudaFuncGetAttributes(&fa, solve_kernel<true, 1024, 1>);
    if (e != cudaSuccess) return e;
    if ((e = set_smem_attr(solve_kernel<true, 1024, 1>, (int)fa.sharedSizeBytes)) != cudaSuccess) return e;
    if ((e = set_smem_attr(solve_kernel<true, 512, 8>, (int)fa.sharedSizeBytes)) != cudaSuccess) return e;
    attr_set = true;
  }
  // Latency path: few scenarios of many jobs leave most of the 148 SMs idle with one CTA per scenario — a cluster of
  // 8 CTAs (portable size, same die) shares one scenario over distributed shared memory instead.
  if (L.jobs_in_smem && L.cluster == 8 && L.J >= 512 && L.S * 8 <= 144) {
    const int Jc = ((((L.J + 7) / 8) + 31) & ~31);
    const size_t smem = smem_fixed + (size_t)Jc * (2 * sizeof(double) + 5 * (size_t)nbases + 3);
    int nt = Jc < 512 ? Jc : 512;
    if (nt < 64) nt = 64;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(L.S * 8)); cfg.blockDim = dim3((unsigned)nt);
    cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = 8; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, solve_kernel<true, 512, 8>, L);
  }
  size_t smem = smem_fixed;
  if (L.jobs_in_smem) smem += (size_t)L.J * (2 * sizeof(double) + 5 * (size_t)nbases + 3);
  int nt = ((L.J + 31) / 32) * 32;
  if (nt > 1024) nt = 1024;
  if (nt < 64) nt = 64;
  if (!L.jobs_in_smem) solve_kernel<false, 1024, 1><<<L.S, nt, smem, st>>>(L);
  else solve_kernel<true, 1024, 1><<<L.S, nt, smem, st>>>(L);
  return cudaGetLastError();
}

}  // namespace swb
