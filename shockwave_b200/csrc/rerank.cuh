// rerank.cuh — local search of the fallback re-rank (rank_in_schedule_jobs, scheduler/shockwave.py:714-793):
// minimise sum_j prio_j * mean round index of job j with the per-job round counts fixed, per-round capacity G.
//
// With w_j = prio_j / n_j the objective is sum_j w_j * sum_{t in rounds(j)} t — a min-cost transportation problem
// (jobs x rounds, a job at most once per round) whose item sizes are the gang widths.  The priority round-sweep of
// place.cu builds a feasible schedule; this pass improves it by NEGATIVE-CYCLE CANCELLING on the round graph:
//   nodes     the T rounds + one slack node
//   edge a->c (a, c rounds) of width class g: the cheapest way to move g GPUs worth of jobs from round a to round c
//             = the job of width g present in a and absent from c with the smallest w_j (c - a), OR (nested widths, the
//             reference's {1,2,4,8} gangs) a composite of two disjoint items of width g/2 — so one 4-gang can trade places
//             with two 2-gangs or a 2-gang and two singles
//   edge slack->a  cost 0 (a round may simply lose a job);  edge c->slack cost 0 if round c has >= g idle GPUs
// A negative cycle of one width class leaves every round's load unchanged (or moves load into idle GPUs through the
// slack node) and lowers the objective by its (negative) cost; for unit widths cancelling until none is left is the
// exact min-cost-flow optimum, for mixed widths it is a local optimum of a neighbourhood that contains every
// same-class exchange chain and the nested cross-class ones.  Per cancelled cycle: one pass over (round pair, job)
// (a thread per ordered pair, the job's round masks broadcast from shared memory) and one Bellman-Ford on <= 129 nodes
// per width class (one warp each, Jacobi sweeps over a dense cost matrix in L2).
// SWAP INTO IDLE GPUs (tried when no negative cycle is left): a job of width 2g moves a -> c while a job of width g moves
// c -> a and round c absorbs the net g GPUs in its idle capacity — the move that lets a wide gang step up into a round
// with fewer idle GPUs than its width (it mixes two width classes AND idle GPUs, so no single-class cycle contains it).
// Multi-start ("noising"): with a seed the first <= 24 cycles are cancelled under weights perturbed by +-30 %, which
// lands the search in another basin; place.cu runs 8 seeds in a thread-block cluster and keeps the best result.
#pragma once
#include "swb_common.cuh"
#include "swb_internal.h"

namespace swb {


#define RR_MAXCLS 4
#define RR_ITEMJOBS 8

// scratch of one search (global memory, L2 resident), carved by rr_carve()
struct RrScratch {
  double *wj;              // [J] w_j = prio_j / n_j (0: job not movable)
  double *cost;            // [RR_MAXCLS][N*N] dense edge costs, N = T + 1, row u -> column v
  unsigned short *jobs;    // [RR_MAXCLS][T*T][RR_ITEMJOBS] jobs of the best item of every (class, pair)
  unsigned char *nj;       // [RR_MAXCLS][T*T] number of jobs of that item
  int *log;                // [(T+1) * RR_ITEMJOBS][2] moves of the cycle being applied: job | from << 16, to
  double *swc;             // [N*N] cost of the best swap-into-idle move of the pair a -> c (1e300: none)
  unsigned short *swj;     // [N*N][4] its jobs (with the edge, against it) and its class
  unsigned long long *bkx; // [J][2] round masks of the best schedule so far (iterated search)
  int *bki;                // [T] its idle GPUs
  double *wn;              // [J] w_j x noise of the current phase (what the edge costs are built from)
  unsigned short *ord;     // [J] movable jobs grouped by width class, ascending job index inside a class
  size_t hot_bytes;        // w_j and the dense cost matrices: the head of the scratch, or of a copy in shared memory
};
#define RR_MAXBAN 64
#define RR_REV 0x8000u     // job entry of an item: this job moves AGAINST the edge (v -> u)
// Carves the scratch of one search at `base` (256-byte aligned) and returns its size, a multiple of 256 bytes.  With
// hot != null (16-byte aligned, hot_bytes long) w_j and the dense cost matrices are read from there instead.
// Called with base = hot = nullptr it only sizes.
__host__ __device__ __forceinline__ size_t rr_carve(RrScratch &s, unsigned char *base, unsigned char *hot, int J,
                                                    int T) {
  const size_t N = (size_t)T + 1, TT = (size_t)T * T;
  unsigned char *p = base;
  s.wj = reinterpret_cast<double *>(p); p += (size_t)J * 8;
  s.cost = reinterpret_cast<double *>(p); p += RR_MAXCLS * N * N * 8;
  s.hot_bytes = (size_t)(p - base);
  s.jobs = reinterpret_cast<unsigned short *>(p); p += RR_MAXCLS * TT * RR_ITEMJOBS * 2;
  s.nj = p; p += RR_MAXCLS * TT;
  p = align16(p);
  s.log = reinterpret_cast<int *>(p); p += N * RR_ITEMJOBS * 8;
  s.swc = reinterpret_cast<double *>(p); p += N * N * 8;
  s.swj = reinterpret_cast<unsigned short *>(p); p += N * N * 8;
  p = align16(p);
  s.bkx = reinterpret_cast<unsigned long long *>(p); p += (size_t)J * 16;
  s.bki = reinterpret_cast<int *>(p); p += N * 4;
  p = align16(p);
  s.wn = reinterpret_cast<double *>(p); p += (size_t)J * 8;
  s.ord = reinterpret_cast<unsigned short *>(p); p += (size_t)J * 2;
  if (hot) {
    s.wj = reinterpret_cast<double *>(hot);
    s.cost = s.wj + J;
  }
  return ((size_t)(p - base) + 255) & ~(size_t)255;
}

__device__ __forceinline__ double rr_noise(int j, unsigned seed) {
  if (seed == 0u) return 1.0;
  unsigned h = (unsigned)j * 0x9E3779B1u ^ seed * 0x85EBCA77u;
  h ^= h >> 15; h *= 0x2C1B3C6Du; h ^= h >> 12; h *= 0x297A2D39u; h ^= h >> 15;
  return 1.0 + 0.3 * ((double)(h & 0xffffffu) * (2.0 / 16777215.0) - 1.0);
}

struct RrItem { double cost; int n; unsigned short job[RR_ITEMJOBS]; };

// Edge costs and best items of every ordered pair of rounds and every width class.  One thread per pair; the inner
// loop over the jobs keeps the two cheapest SINGLE jobs per class in registers (cls_of[] maps a width to its class).
__device__ void rr_build(const RrScratch &S, const unsigned long long *xm, const int *off,
                         const int *clsw, int ncls, const int *idle, int J, int T) {
  const double INF = 1e300;
  const int N = T + 1;
  for (int pr = threadIdx.x; pr < N * N; pr += blockDim.x) {
    const int a = pr / N, c = pr - a * N;
    if (a == T || c == T || a == c) {
      // slack edges and the diagonal
      for (int k = 0; k < ncls; ++k) {
        double v = INF;
        if (a == T && c != T) v = 0.0;
        else if (c == T && a != T) v = (idle[a] >= clsw[k]) ? 0.0 : INF;
        S.cost[(size_t)k * N * N + pr] = v;
      }
      S.swc[pr] = INF;
      continue;
    }
    double c0[RR_MAXCLS], c1[RR_MAXCLS], cr[RR_MAXCLS];      // cr / jr: cheapest single job moving c -> a (against the edge)
    int j0[RR_MAXCLS], j1[RR_MAXCLS], jr[RR_MAXCLS];
    const int wa = a >> 6, wc = c >> 6;
    const unsigned long long ba = 1ull << (a & 63), bc = 1ull << (c & 63);
    const double dist = (double)(c - a);
    // one pass per width class over THAT class's jobs (S.ord, ascending job index = the order of the plain loop, so
    // ties break the same way): the class is a compile-time index, the running best / second best are scalars —
    // ncu r02: the one-loop form with a 4-way class select spent ~60 instructions per (pair, job) and the per-thread
    // chain of the rebuild was the critical path of every search iteration
#pragma unroll
    for (int k = 0; k < RR_MAXCLS; ++k) {
      double b0 = INF, b1 = INF, br = INF;
      int i0 = -1, i1 = -1, ir = -1;
      if (k < ncls) {
        for (int i = off[k]; i < off[k + 1]; ++i) {
          const int j = S.ord[i];
          const bool ina = (xm[2 * j + wa] & ba) != 0ull, inc = (xm[2 * j + wc] & bc) != 0ull;
          if (ina == inc) continue;
          const double x = S.wn[j] * dist;
          if (ina) {
            if (x < b0) { b1 = b0; i1 = i0; b0 = x; i0 = j; }
            else if (x < b1) { b1 = x; i1 = j; }
          } else if (-x < br) { br = -x; ir = j; }
        }
      }
      c0[k] = b0; c1[k] = b1; cr[k] = br; j0[k] = i0; j1[k] = i1; jr[k] = ir;
    }
    // best / second-best ITEM per class: singles, plus the composite of the two best items of half the width
    RrItem b0, b1;                       // of the previous class
    b0.cost = INF; b0.n = 0; b1.cost = INF; b1.n = 0;
    const int tp = a * T + c;
#pragma unroll
    for (int k = 0; k < RR_MAXCLS; ++k) {
      if (k >= ncls) break;
      RrItem n0, n1;
      n0.cost = c0[k]; n0.n = j0[k] >= 0 ? 1 : 0; n0.job[0] = (unsigned short)j0[k];
      n1.cost = c1[k]; n1.n = j1[k] >= 0 ? 1 : 0; n1.job[0] = (unsigned short)j1[k];
      if (k > 0 && clsw[k] == 2 * clsw[k - 1] && b1.cost < INF && b0.n + b1.n <= RR_ITEMJOBS) {
        RrItem x;
        x.cost = b0.cost + b1.cost; x.n = b0.n + b1.n;
        for (int q = 0; q < b0.n; ++q) x.job[q] = b0.job[q];
        for (int q = 0; q < b1.n; ++q) x.job[b0.n + q] = b1.job[q];
        bool dup = false;                  // items that contain a swap can share a job: not a valid composite
        for (int q = 0; q < b0.n; ++q)
          for (int r = 0; r < b1.n; ++r) dup |= ((b0.job[q] ^ b1.job[r]) & 0x7fffu) == 0u;
        if (!dup) { if (x.cost < n0.cost) { n1 = n0; n0 = x; } else if (x.cost < n1.cost) n1 = x; }
      }
      S.cost[(size_t)k * N * N + pr] = n0.cost;
      S.nj[(size_t)k * T * T + tp] = (unsigned char)n0.n;
      for (int q = 0; q < n0.n; ++q) S.jobs[((size_t)k * T * T + tp) * RR_ITEMJOBS + q] = n0.job[q];
      b0 = n0; b1 = n1;
    }
    // swap into idle GPUs: a job of class k+1 (twice the width) a -> c, a job of class k c -> a, round c takes the net
    // width of class k out of its idle GPUs
    double sb = INF;
    int sk = 0, sA = 0, sB = 0;
#pragma unroll
    for (int k = 0; k + 1 < RR_MAXCLS; ++k) {
      if (k + 1 >= ncls) break;
      if (clsw[k + 1] != 2 * clsw[k] || j0[k + 1] < 0 || jr[k] < 0 || idle[c] < clsw[k]) continue;
      const double x = c0[k + 1] + cr[k];
      if (x < sb) { sb = x; sk = k; sA = j0[k + 1]; sB = jr[k]; }
    }
    S.swc[pr] = sb;
    S.swj[4 * pr] = (unsigned short)sA; S.swj[4 * pr + 1] = (unsigned short)sB; S.swj[4 * pr + 2] = (unsigned short)sk;
  }
}

// One warp: Bellman-Ford (Jacobi sweeps, double-buffered distances) from a virtual source on one class's dense cost
// matrix; returns the length of a negative cycle written to cyc[] (nodes in forward order), 0 if there is none.
__device__ int rr_find_cycle(const double *cost, int T, double *d, short *pred, short *cyc, double tol) {
  const int lane = threadIdx.x & 31, N = T + 1;
  const double INF = 1e300;
  double *dold = d, *dnew = d + (SWB_MAX_T + 1);
  for (int v = lane; v < N; v += 32) { dold[v] = 0.0; dnew[v] = 0.0; pred[v] = -1; }
  __syncwarp();
  int last = -1;
  for (int it = 0; it < N; ++it) {
    int changed = -1;
    for (int v = lane; v < N; v += 32) {
      double dv = dold[v];
      int pv = -2;
      for (int u = 0; u < N; ++u) {
        const double cuv = cost[u * N + v];
        if (cuv >= INF * 0.5) continue;
        const double cand = dold[u] + cuv;
        if (cand < dv - tol) { dv = cand; pv = u; }
      }
      dnew[v] = dv;
      if (pv != -2) { pred[v] = (short)pv; changed = v; }
    }
    changed = __reduce_max_sync(SWB_FULL, changed);
    __syncwarp();
    double *t = dold; dold = dnew; dnew = t;
    last = changed;
    if (changed < 0) return 0;
    // A negative cycle shows up in the predecessor graph long before the N-th sweep: every 4th sweep (and at the
    // end) walk back from the last relaxed node; a node met twice closes a cycle, which is returned if its cost is
    // negative (the caller re-verifies with compensated summation).
    if ((it & 3) == 3 || it == N - 1) {
      int len = 0;
      if (lane == 0) {
        int x = last;
        for (int q = 0; q < N && x >= 0; ++q) x = pred[x];
        if (x >= 0) {
          int cur = x, guard = 0;
          double tot = 0.0;
          do {
            cyc[len++] = (short)cur;
            const int pu = pred[cur];
            if (pu < 0) break;
            tot += cost[pu * N + cur];
            cur = pu;
          } while (cur != x && ++guard <= N);
          if (cur != x || !(tot < -tol)) len = 0;
          for (int q = 0; q < len / 2; ++q) { const short t2 = cyc[q]; cyc[q] = cyc[len - 1 - q]; cyc[len - 1 - q] = t2; }
        }
      }
      len = __shfl_sync(SWB_FULL, len, 0);
      __syncwarp();
      if (len >= 2) return len;
    }
  }
  return 0;
}

// sum_j w_j * (sum of the round indices of job j); every thread gets the result.  part: 32 doubles of shared scratch.
__device__ double rr_objective(const RrScratch &S, const unsigned long long *xm, int J, double *part) {
  double acc = 0.0;
  for (int j = threadIdx.x; j < J; j += blockDim.x) {
    const double w = S.wj[j];
    if (w == 0.0) continue;
    int st = 0;
    for (int wi = 0; wi < 2; ++wi) {
      unsigned long long m = xm[2 * j + wi];
      while (m) { st += 64 * wi + (__ffsll((long long)m) - 1); m &= m - 1; }
    }
    acc += w * (double)st;
  }
  acc = warp_sum(acc);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = acc;
  __syncthreads();
  double tot = 0.0;
  for (int q = 0; q < (int)((blockDim.x + 31) >> 5); ++q) tot += part[q];
  __syncthreads();
  return tot;
}

// The local search.  All threads of the CTA call it.  xm: [J][2] round masks (in/out); idle: [T] (in/out).
// Returns the number of cancelled cycles; *final_cost = objective of the result under the true weights.
__device__ __noinline__ int rr_local_search(unsigned char *scratch, unsigned char *hot, unsigned long long *xm,
                                            const unsigned char *gs,
                                            const unsigned char *remn, const unsigned char *nplan, const double *prio,
                                            int *idle, int J, int T, int max_iters, unsigned noise_seed,
                                            int restarts, double *final_cost) {
  __shared__ double ws_d[RR_MAXCLS * 2 * (SWB_MAX_T + 1)];
  __shared__ short ws_pred[RR_MAXCLS * (SWB_MAX_T + 1)];
  __shared__ short ws_cyc[RR_MAXCLS * (SWB_MAX_T + 2)];
  __shared__ unsigned char s_clsof[256];
  __shared__ int s_cls[RR_MAXCLS], s_ncls, s_found, s_len[RR_MAXCLS], s_ban[RR_MAXBAN], s_nban, s_off[RR_MAXCLS + 1];
  __shared__ double s_part[32];
  __shared__ int s_parti[32];
  RrScratch S;
  rr_carve(S, scratch, hot, J, T);
  const int N = T + 1;
  for (int j = threadIdx.x; j < J; j += blockDim.x)
    S.wj[j] = (nplan[j] > 0 && remn[j] == 0 && isfinite(prio[j])) ? prio[j] / (double)nplan[j] : 0.0;
  for (int i = threadIdx.x; i < 256; i += blockDim.x) s_clsof[i] = 255;
  __syncthreads();
  if (threadIdx.x == 0) {
    // width classes: the (up to 4) distinct widths among the placed jobs, ascending
    int n = 0, w[RR_MAXCLS];
    for (int j = 0; j < J; ++j) {
      if (nplan[j] == 0) continue;
      const int g = gs[j];
      bool seen = false;
      for (int q = 0; q < n; ++q) seen |= (w[q] == g);
      if (!seen) { if (n == RR_MAXCLS) { n = RR_MAXCLS + 1; break; } w[n++] = g; }
    }
    if (n > RR_MAXCLS) n = 0;                     // more than 4 distinct widths: leave the sweep's schedule as it is
    for (int q = 1; q < n; ++q) for (int r = q; r > 0 && w[r - 1] > w[r]; --r) { int t = w[r]; w[r] = w[r - 1]; w[r - 1] = t; }
    for (int q = 0; q < n; ++q) { s_cls[q] = w[q]; s_clsof[w[q]] = (unsigned char)q; }
    s_ncls = n;
    s_nban = 0;
    // movable jobs grouped by class (counting sort, ascending job index inside a class)
    int cnt[RR_MAXCLS + 1];
    for (int q = 0; q <= RR_MAXCLS; ++q) cnt[q] = 0;
    for (int j = 0; j < J; ++j) if (n > 0 && S.wj[j] != 0.0 && s_clsof[gs[j]] < RR_MAXCLS) ++cnt[s_clsof[gs[j]] + 1];
    for (int q = 0; q < RR_MAXCLS; ++q) cnt[q + 1] += cnt[q];
    for (int q = 0; q <= RR_MAXCLS; ++q) s_off[q] = cnt[q];
    for (int j = 0; j < J; ++j)
      if (n > 0 && S.wj[j] != 0.0 && s_clsof[gs[j]] < RR_MAXCLS) S.ord[cnt[s_clsof[gs[j]]]++] = (unsigned short)j;
  }
  __syncthreads();
  const int ncls = s_ncls;
  if (ncls == 0) { if (threadIdx.x == 0) *final_cost = 1e300; __syncthreads(); return 0; }
  // scale of the tolerances: the CURRENT objective (not the largest weight: a job whose priority is 1e12 times the
  // others' sits in round 0 and contributes nothing, while exchanges among the ordinary jobs still move the objective)
  const double scale = fmax(rr_objective(S, xm, J, s_part), 1e-300);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  int done = 0;
  // ITERATED local search: after the first local optimum the search is perturbed again (a fresh noise seed, from the
  // best schedule so far) `restarts` times; a round that does not improve is undone.
  double best_cost = 1e300;
  for (int rs = 0; rs <= restarts; ++rs) {
  const unsigned seed_rs = rs == 0 ? noise_seed : (noise_seed * 2654435761u + (unsigned)rs * 40503u + 977u) | 1u;
  if (threadIdx.x == 0) s_nban = 0;
  __syncthreads();
  // phase 0 (only with a noise seed): up to 24 cycles under perturbed weights, to reach another basin;
  // phase 1: true weights until no negative cycle is left (or the budget is spent)
  int phase = seed_rs ? 0 : 1, phase_iters = 0, wn_phase = -1;
  for (int iter = 0; iter < max_iters; ++iter) {
    if (phase != wn_phase) {                   // edge costs use w_j x noise(phase): once per phase, not per (pair, job)
      const unsigned sd = phase == 0 ? seed_rs : 0u;
      for (int j = threadIdx.x; j < J; j += blockDim.x) S.wn[j] = S.wj[j] * rr_noise(j, sd);
      wn_phase = phase;
      __syncthreads();
    }
    rr_build(S, xm, s_off, s_cls, ncls, idle, J, T);
    if (threadIdx.x == 0) s_found = -1;
    __syncthreads();
    if ((int)threadIdx.x < s_nban) S.cost[(size_t)(s_ban[threadIdx.x] >> 28) * N * N + (s_ban[threadIdx.x] & 0xfffffff)] = 1e300;
    __syncthreads();
    for (int k = warp; k < ncls; k += (int)(blockDim.x >> 5)) {       // one warp per width class
      const int len = rr_find_cycle(S.cost + (size_t)k * N * N, T, ws_d + k * 2 * (SWB_MAX_T + 1),
                                    ws_pred + k * (SWB_MAX_T + 1), ws_cyc + k * (SWB_MAX_T + 2), 1e-11 * scale);
      if (lane == 0) s_len[k] = len;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      // the lowest class that has a cycle; verify it is really negative (tolerances) and apply it
      for (int k = 0; k < ncls && s_found < 0; ++k) {
        const int len = s_len[k];
        if (len < 2) continue;
        const short *cyc = ws_cyc + k * (SWB_MAX_T + 2);
        const double *ck = S.cost + (size_t)k * N * N;
        // gain of the cycle, Neumaier-compensated: edge costs span many decades and a huge +X / -X pair must
        // cancel exactly instead of leaving rounding noise that looks like an improvement
        double tot = 0.0, comp = 0.0;
        bool ok = true;
        for (int q = 0; q < len && ok; ++q) {
          const int u = cyc[q], v = cyc[(q + 1) % len];
          const double x = ck[u * N + v];
          if (x >= 1e299) { ok = false; break; }
          const double t2 = tot + x;
          comp += (fabs(tot) >= fabs(x)) ? (tot - t2) + x : (x - t2) + tot;
          tot = t2;
        }
        tot += comp;
        if (!ok || !(tot < -1e-11 * scale)) continue;
        // apply the cycle job by job with its precondition (present in the source round, absent from the target):
        // items that mix classes can name the same job on two edges of one cycle; such a cycle is rolled back and its
        // first offending edge is banned for the rest of the search (s_ban)
        int nlog = 0, bad_edge = -1;
        for (int q = 0; q < len && bad_edge < 0; ++q) {
          const int u = cyc[q], v = cyc[(q + 1) % len];
          if (u == T || v == T) continue;
          const size_t tp = (size_t)k * T * T + (size_t)u * T + v;
          const int nj = S.nj[tp];
          for (int e = 0; e < nj; ++e) {
            const unsigned int raw = S.jobs[tp * RR_ITEMJOBS + e];
            const int j = (int)(raw & 0x7fffu);
            const int from = (raw & RR_REV) ? v : u, to = (raw & RR_REV) ? u : v;
            const unsigned long long bf = 1ull << (from & 63), bt2 = 1ull << (to & 63);
            if (!(xm[2 * j + (from >> 6)] & bf) || (xm[2 * j + (to >> 6)] & bt2)) { bad_edge = u * N + v; break; }
            xm[2 * j + (from >> 6)] &= ~bf;
            xm[2 * j + (to >> 6)] |= bt2;
            S.log[2 * nlog] = j | (from << 16); S.log[2 * nlog + 1] = to; ++nlog;
          }
        }
        if (bad_edge >= 0) {
          for (int q = nlog - 1; q >= 0; --q) {
            const int j = S.log[2 * q] & 0xffff, from = S.log[2 * q] >> 16, to = S.log[2 * q + 1];
            xm[2 * j + (to >> 6)] &= ~(1ull << (to & 63));
            xm[2 * j + (from >> 6)] |= 1ull << (from & 63);
          }
          if (s_nban < RR_MAXBAN) { s_ban[s_nban] = (k << 28) | bad_edge; s_nban = s_nban + 1; s_found = -2; }
          continue;
        }
        for (int q = 0; q < len; ++q) {
          const int u = cyc[q], v = cyc[(q + 1) % len];
          if (u == T) idle[v] += s_cls[k];                          // v loses an item that no cycle edge brings back
          else if (v == T) idle[u] -= s_cls[k];                     // u keeps an item: its idle GPUs take it
        }
        s_found = k;
      }
    }
    __syncthreads();
    if (s_found == -1) {
      // no negative cycle: the best swap-into-idle move of any ordered pair of rounds (block arg-min, lowest pair wins ties)
      double bv = -1e-11 * scale;
      int bi = -1;
      for (int pr = threadIdx.x; pr < N * N; pr += blockDim.x) {
        const double v = S.swc[pr];
        if (v < bv) { bv = v; bi = pr; }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const double ov = __shfl_xor_sync(SWB_FULL, bv, o);
        const int oi = __shfl_xor_sync(SWB_FULL, bi, o);
        if (oi >= 0 && (bi < 0 || ov < bv || (ov == bv && oi < bi))) { bv = ov; bi = oi; }
      }
      if (lane == 0) { s_part[warp] = bv; s_parti[warp] = bi; }
      __syncthreads();
      if (threadIdx.x == 0) {
        double gv = 0.0;
        int gi = -1;
        for (int q = 0; q < (int)((blockDim.x + 31) >> 5); ++q) {
          const int oi = s_parti[q];
          if (oi >= 0 && (gi < 0 || s_part[q] < gv || (s_part[q] == gv && oi < gi))) { gv = s_part[q]; gi = oi; }
        }
        if (gi >= 0) {
          const int a = gi / N, c2 = gi - a * N;
          const int A = S.swj[4 * gi], B = S.swj[4 * gi + 1], k = S.swj[4 * gi + 2];
          const unsigned long long ba = 1ull << (a & 63), bc = 1ull << (c2 & 63);
          const bool okA = (xm[2 * A + (a >> 6)] & ba) && !(xm[2 * A + (c2 >> 6)] & bc);
          const bool okB = (xm[2 * B + (c2 >> 6)] & bc) && !(xm[2 * B + (a >> 6)] & ba);
          if (okA && okB && idle[c2] >= s_cls[k]) {
            xm[2 * A + (a >> 6)] &= ~ba; xm[2 * A + (c2 >> 6)] |= bc;
            xm[2 * B + (c2 >> 6)] &= ~bc; xm[2 * B + (a >> 6)] |= ba;
            idle[c2] -= s_cls[k]; idle[a] += s_cls[k];
            s_found = RR_MAXCLS;                   // "a move was applied"
          }
        }
      }
      __syncthreads();
    }
    ++phase_iters;
    if (s_found == -2) continue;                 // a cycle was rolled back and its edge banned: search again
    if (phase == 0 && (s_found < 0 || phase_iters >= 24)) { phase = 1; continue; }
    if (s_found < 0) break;
    ++done;
  }
  const double fc_rs = rr_objective(S, xm, J, s_part);
  if (restarts > 0) {
    if (fc_rs < best_cost) {                     // keep
      best_cost = fc_rs;
      for (int i = threadIdx.x; i < 2 * J; i += blockDim.x) S.bkx[i] = xm[i];
      for (int i = threadIdx.x; i < T; i += blockDim.x) S.bki[i] = idle[i];
    } else {                                     // undo this round
      for (int i = threadIdx.x; i < 2 * J; i += blockDim.x) xm[i] = S.bkx[i];
      for (int i = threadIdx.x; i < T; i += blockDim.x) idle[i] = S.bki[i];
    }
    __syncthreads();
  }
  }
  const double fc = rr_objective(S, xm, J, s_part);
  if (threadIdx.x == 0) *final_cost = fc;
  __syncthreads();
  return done;
}

}  // namespace swb
