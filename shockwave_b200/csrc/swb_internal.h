// Internal launch descriptors shared by the .cu files of libswb200 (not part of the C-ABI).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>

#include "../../include/swb200.h"

#define SWB_SOLVE_THREADS 1024
#define SWB_PLACE_THREADS 1024
#define SWB_SMEM_JOBS 4096          /* job constants staged in shared memory up to this J */
#define SWB_PWL_BYTES 512           /* >= sizeof(swb::Pwl), 16-byte aligned */
#define SWB_MAX_DYN_SMEM (227 * 1024)
#define SWB_MAX_T 128               /* x rows are kept as 128-bit masks in the placement kernel */
#define SWB_MAX_REPLAN 6             /* packing-feedback re-solves (caps written by place_kernel) */
#define SWB_MAX_J 8192              /* 13 index bits in the placement sort key */

// sets swb_last_error() and returns `code`
extern "C" int swb_set_error(int code, const char *msg);

// return SWB_ERR_CUDA from the enclosing entry point when a CUDA call fails
#define CK(call)                                                                                   \
  do {                                                                                             \
    cudaError_t e_ = (call);                                                                       \
    if (e_ != cudaSuccess)                                                                         \
      return swb_set_error(SWB_ERR_CUDA, (std::string(#call) + ": " + cudaGetErrorString(e_)).c_str()); \
  } while (0)

// capacity after growing `cap` to hold `bytes`: doubling from 256 bytes
inline size_t swb_grow_cap(size_t cap, size_t bytes) {
  size_t ncap = cap ? cap : 256;
  while (ncap < bytes) ncap *= 2;
  return ncap;
}

// Grow-only device buffer, freed by its destructor.  need() with `keep` preserves the old contents and zeroes the
// new tail (the resident job table grows in place that way); without it the contents are undefined after growth.
struct DBuf {
  void *p = nullptr;
  size_t cap = 0;
  DBuf() = default;
  DBuf(const DBuf &) = delete;
  DBuf &operator=(const DBuf &) = delete;
  ~DBuf() { if (p) cudaFree(p); }
  cudaError_t need(size_t bytes, cudaStream_t st, bool keep = false) {
    if (bytes <= cap) return cudaSuccess;
    const size_t ncap = swb_grow_cap(cap, bytes);
    void *np = nullptr;
    cudaError_t e = cudaMalloc(&np, ncap);
    if (e != cudaSuccess) return e;
    if (keep && p && cap) {
      e = cudaMemcpyAsync(np, p, cap, cudaMemcpyDeviceToDevice, st);
      if (e != cudaSuccess) return e;
      e = cudaStreamSynchronize(st);
      if (e != cudaSuccess) return e;
    }
    if (keep && ncap > cap) {
      e = cudaMemsetAsync((char *)np + cap, 0, ncap - cap, st);
      if (e != cudaSuccess) return e;
    }
    if (p) cudaFree(p);
    p = np; cap = ncap;
    return cudaSuccess;
  }
  // grow to `bytes`, then copy `bytes` from the host on `st`
  cudaError_t upload(const void *src, size_t bytes, cudaStream_t st) {
    const cudaError_t e = need(bytes, st);
    return e != cudaSuccess ? e : cudaMemcpyAsync(p, src, bytes, cudaMemcpyHostToDevice, st);
  }
  template <class T> T *as() { return reinterpret_cast<T *>(p); }
};

// Grow-only pinned host buffer (staging of truly asynchronous copies), freed by its destructor; the contents are
// undefined after growth.
struct PinBuf {
  void *p = nullptr;
  size_t cap = 0;
  PinBuf() = default;
  PinBuf(const PinBuf &) = delete;
  PinBuf &operator=(const PinBuf &) = delete;
  ~PinBuf() { if (p) cudaFreeHost(p); }
  cudaError_t need(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    const size_t ncap = swb_grow_cap(cap, bytes);
    if (p) cudaFreeHost(p);
    p = nullptr; cap = 0;
    const cudaError_t e = cudaMallocHost(&p, ncap);
    if (e == cudaSuccess) cap = ncap;
    return e;
  }
  template <class T> T *as() { return reinterpret_cast<T *>(p); }
};

namespace swb {

struct SolveLaunch {
  int S, J, per_scn, jobs_in_smem;
  const swb_params *prm;  // device [S]
  const int32_t *g, *E, *c;
  const double *dbar, *rem, *ftobj;
  const double *rem_fb;   // remaining runtime as seen by relax_finish_time_constraints (may be null -> rem)
  // per-scenario scratch in global memory, [S][J]
  double *sc_a, *sc_u0, *sc_R, *sc_ws, *sc_cap;
  uint8_t *sc_g, *sc_nF, *sc_nmax, *sc_n;
  // response table in global memory, only used when J > SWB_SMEM_JOBS ([S][J] and [S][J][SWB_MAX_BASES])
  double *sc_cth, *sc_Rr;   // sc_Rr: remaining runtime in rounds (the table copy; sc_R keeps seconds)
  float *sc_ths;
  uint8_t *sc_n0;
  double *sc_nfc;      // [S][J] continuous FTF lower bounds (relaxation only)
  int want_relaxed;    // also compute the exact optimum of the continuous relaxation (slow; parity item P4)
  const uint8_t *ncap; // [S][J] per-job cap on the round count from packing feedback (255 = none)
  double *weights;   // [S][J] out, may be null
  swb_result *res;   // device [S]
  int cluster;       // SWB_OPT_SOLVE_CLUSTER: 8 lets few scenarios of many jobs share each over a cluster of 8 CTAs
};

// How one call's placement is launched, decided once by plan_place (place.cu).
struct PlacePlan {
  int rerank;             // 1: the fallback re-rank search runs
  int cluster;            // CTAs per scenario: 8 (the search starts from 8 seeds over a thread-block cluster) or 1
  int hot_smem;           // 1: the search's hot arrays (w_j, dense edge costs) sit in shared memory, 0: in its scratch
  int threads;            // per CTA
  size_t smem;            // dynamic shared memory per CTA
  size_t rr_region;       // scratch of one search
  size_t rr_bytes;        // scratch of the launch: S x cluster regions (0: search off)
};
PlacePlan plan_place(int S, int J, int T, int rr_iters, int cluster_opt);

struct PlaceLaunch {
  int S, J, per_scn;
  const swb_params *prm;  // device [S]
  const double *bfkey;    // [S][J] or [J]
  const double *bfkey_fb; // same, for the fallback continuation (may be null -> bfkey)
  const double *sc_a, *sc_u0, *sc_R, *sc_ws, *sc_cap;
  const uint8_t *sc_g, *sc_n, *sc_nmax;
  const double *weights;  // [S][J] (priority, for the fallback re-rank), may be null
  const int32_t *E, *c;   // solver inputs again (objective re-evaluation with the checker's formula)
  const double *dbar;
  uint8_t *x, *backfill;  // [S][J][T] out, may be null
  unsigned long long *xmask, *bfmask;  // [S][J][2] out, may be null: bit t of the 128-bit row = round t
  int32_t *nrounds;       // [S][J] out, may be null
  int32_t *ncal;          // [S][J] out, may be null: rounds with idle GPUs in which the job is unscheduled
  swb_result *res;        // device [S] (status in, objective/shortfall updated)
  uint8_t *ncap;          // [S][J] in/out, may be null: per-job count caps for the next pass (packing feedback)
  void *rr_items;         // scratch of the re-rank local search, plan.rr_bytes
  int rr_iters;           // cycle-cancelling budget per scenario
  int rr_restarts;        // perturb-and-continue rounds after the first local optimum (iterated local search)
  PlacePlan plan;
};

cudaError_t launch_solve(const SolveLaunch &L, cudaStream_t st, int nbases);
cudaError_t launch_place(const PlaceLaunch &L, cudaStream_t st, unsigned long long *gmask);

struct ForecastLaunch {
  int J;
  int reestimate_share;
  int round_ptr, ngpus;
  double gavel_round_duration;
  // per-call inputs [J]
  const int32_t *slots, *progress, *meas_end;
  const double *meas_ns;
  // resident job table (indexed by slot)
  const int64_t *tab_off;       // start of the job's rows in the pools (E+1 rows per job in both)
  const int32_t *tab_E, *tab_nmodes, *tab_g;
  const double *tab_nsamples, *tab_tsubmit;
  const int32_t *tab_modes;     // [slot][SWB_MAX_MODES]
  const double *tab_modemean;   // [slot][SWB_MAX_MODES] mean pre-profiled duration per bs mode
  double *tab_amp;              // calibration factor state (JobMetaData.py:281-286)
  // share-series state (shockwave.py:114-118, :480-501): first round, last round, last value,
  // running sum of gap*value, number of entries
  int32_t *ss_r0, *ss_rlast, *ss_cnt;
  double *ss_vlast, *ss_acc;
  const double *pool_prefix;    // prefix sums of the pre-profiled epoch durations (E+1 per job)
  const int32_t *pool_bs;       // bs_schedule (E per job)
  // outputs [J]
  double *dbar, *rem, *ftobj, *bfkey, *ftest;
  double *rem_fb, *bfkey_fb, *amp_ok, *amp_fb;
  int32_t *g_out, *E_out, *c_out;
};
cudaError_t launch_forecast(const ForecastLaunch &L, cudaStream_t st);
cudaError_t launch_commit_calibration(const ForecastLaunch &L, const swb_result *res, int fallback_host,
                                      const int32_t *ncal, cudaStream_t st);

struct PolicyLaunch {
  int mode, J;
  double N;                 // pooled worker count
  const double *coef;       // MAXMIN: thr*sf*priority ; FTF/MTD: throughput ; MAXSUM: thr/cost ; ISOLATED: divisor
  const double *sf;         // scale factors
  const double *t, *n, *den;// FTF: times_since_start, steps remaining, isolated-time denominators ; MTD: n
  double *x;                // [J] out
  double *out;              // [2] out: objective, status
};
cudaError_t launch_policy(const PolicyLaunch &L, cudaStream_t st);

struct HeteroLaunch {
  int mode, J, W;           // SWB_POL_MAXMIN / FTF / MTD / MAXSUM, jobs, worker types (<= 3)
  const double *N;          // [W] workers per type (device)
  const double *a;          // [J][W] MAXMIN: objective coefficients ; FTF/MTD: throughputs ; MAXSUM: thr/cost
  const double *sf;         // [J] scale factors
  const double *t, *n, *den;// as in PolicyLaunch
  double *x;                // [J][W] out
  double *out;              // [4] out: objective, status, pricing passes, feasibility checks
  // water-filling iteration (SWB_POL_WFILL / SWB_POL_WFZ): t = normalised lower bounds, n = multiplicative terms
  // (0: the job takes no part), den = proportional throughputs
  double wf_M = 0.0, wf_slack = 1.0;   // cap of the LP objective; slack factor of the bottleneck test
  const double *wf_c = nullptr;        // WFZ: device pointer to the LP step's objective (lower_j += c / mult_j)
  double *zout = nullptr;              // WFZ: [J] relaxed z_j
};
cudaError_t launch_hetero(const HeteroLaunch &L, cudaStream_t st);

struct AssignLaunch {
  int m, n, W;              // jobs, workers, worker types
  const double *p;          // [m][W] processing time of job i on a worker of type w (steps / throughput)
  const double *t;          // [m] times_since_start
  const int32_t *wtype;     // [n] type of worker j
  double *u, *v, *spc;      // duals [m], [m*n]; shortest-path costs [m*n]
  int32_t *col4row, *row4col, *path;
  unsigned char *inSC, *inSR;
  double *out;              // [1] total cost
};
cudaError_t launch_assign(const AssignLaunch &L, cudaStream_t st);

#define SWB_MK_MAXW 4
struct MarketLaunch {
  int S, J, W, T, per_scn, jobs_per_cta;
  int Tfull;                      // planning rounds of the full problem: objective 1/(J Tfull), makespan in units of D Tfull
  float rscale;                   // progress of one tensor entry = rscale * rate (Tfull/T on the time-coarsened level)
  const swb_params *prm;          // device [S]
  const int32_t *g;               // [J] or [S][J]
  const double *E, *c, *dbar, *rem;
  const float *rate;              // [J][W] or [S][J][W]: epochs of progress per round on worker type w
  const float *icap;              // [W][T] 1 / workers of type w in round t (shared by the scenarios)
  float *X;                       // [S][J][W][T]
  float4 *jobpack;                // [S][J] (theta = gain per unit rate, beta = step-size term, g, rate on type 0)
  float *rowp, *rowprev;          // [S][J]: row reductions of x^{k+1} / x^k
  double *mj, *om;                // [S][J] duals: marginal utility, makespan multipliers
  float *colload, *colprev, *colscale, *price;  // [S][W][T]; price = pi * icap
  double *pi;                     // [S][W][T] capacity prices (normalised rows)
  double *obj;                    // [S][3]: objective, makespan, worst relative capacity violation
  float pw;                       // primal weight asked for (tau = tau0 / pw, sigma = sigma0 * pw)
  float *pws;                     // [S] primal weight in use (market_dual_kernel phase 0: pw raised with k)
  int phase;                      // dual pass: 0 start, 1 PDHG dual step, 2 repair factors, 3 score only
  int mode;                       // dense pass: 0 primal step, 1 column scaling
  int utility;                    // 0: Shockwave's PWL log + makespan term, 1: Eisenberg-Gale sum_j log(U_j)
};
cudaError_t launch_market_prolong(const float *Xc, float *X, const double *pic, double *pi, size_t rows, int S, int W,
                                  int T, int grp, cudaStream_t st);
cudaError_t launch_market_restrict(const float *X, float *Xc, size_t rows, int T, int grp, cudaStream_t st);
cudaError_t launch_market_fill(float *p, size_t n, float v, cudaStream_t st);
cudaError_t launch_market_iter(const MarketLaunch &L, cudaStream_t st, bool dense);

// Gavel's per-round priority -> selection -> worker assignment (gavel.cu).  Worker types appear in PROCESSING order
// in type_order / nworkers / worker_ids; alloc etc. are [J][W] indexed by the caller's type index.
struct GavelLaunch {
  int J, W, flags, maxw;          // flags: bit0 Isolated_plus (strict order), bit1 FIFO (skip priority <= 0)
  const int32_t *type_order;      // [W] type index processed ti-th
  const int32_t *capacity;        // [W] by type index: cluster_spec
  const double *alloc, *job_time, *deficit, *thr;   // [J][W]; alloc = NaN when the job is not in the allocation
  const double *worker_time;      // [W]
  const uint8_t *in_alloc;        // [J]
  const int32_t *sf;              // [J] scale factors
  const int32_t *nworkers;        // [W] by processing position
  const int32_t *worker_ids;      // workers by processing position, server order
  const int32_t *prev_type;       // [J] type index of last round's assignment, -1 = none
  const int32_t *prev_off;        // [J+1]
  const int32_t *prev_local;      // last round's workers as positions in their type's worker list
  double *prio;                   // [J][W] out
  int32_t *n_sel, *sel_jobs;      // [W], [W][J] out: selected jobs per processing position, selection order
  int32_t *assign_job, *assign_cnt, *assign_off, *assign_workers;   // out: assignments in insertion order
  int32_t *tmp_rank0, *tmp_free;  // scratch
  uint8_t *sched;                 // [J] scratch
  int32_t *out_scalars;           // [2]: number of assignments, error flag
};
cudaError_t launch_gavel_round(const GavelLaunch &L, cudaStream_t st);

struct GbmLaunch {
  int J;
  long long P_local, path_offset;
  unsigned long long seed;
  const double *R0, *mu, *sigma;
  const int32_t *H;
  double *out;   // [2][J]: sum R, sum R^2 over the local paths
  // table-driven variant (swb_round_solve): mu / sigma come from the resident job table through `slots`, the
  // horizon is min(E - c, Hmax) from the forecast kernel's own outputs; null -> the plain arrays above
  const int32_t *slots, *Eo, *co;
  const double *tab_mu, *tab_sigma;
  int Hmax;
};
cudaError_t launch_gbm(const GbmLaunch &L, cudaStream_t st);
// rem / bfkey (both continuations) *= E_mc[R] / R0 for the jobs whose model has drift or volatility; jobs with
// mu = sigma = 0 keep the deterministic forecast bit for bit
struct GbmApplyLaunch {
  int J;
  double P_total;
  const double *sums;      // [2][J] after the allreduce
  const int32_t *slots;
  const double *tab_mu, *tab_sigma;
  double *rem, *rem_fb, *bfkey, *bfkey_fb;   // in/out, may be null
  double *var_out;         // [J] variance of the forecast, may be null
};
cudaError_t launch_gbm_apply(const GbmApplyLaunch &L, cudaStream_t st);
// scenario ensemble from one Monte-Carlo forecast: rem[s][j] = max(0, mean_j + z_s * std_j)  (forecast quantiles)
cudaError_t launch_gbm_ensemble(int S, int J, double P_total, const double *sums, const double *z, double *rem_out,
                                cudaStream_t st);

// batch of S linear programs  max c'x : A x <= b, x >= 0  with a shared CSC pattern (lp.cu / lp_core.cuh)
struct LpLaunch {
  int S, m, n, nnz, max_iter;
  const int *colp, *rowi;        // [n + 1], [nnz]  shared by the batch
  const double *val, *c, *b;     // [S][nnz], [S][n], [S][m]
  double *Binv, *Bm;             // [S][m * m] each
  double *vec;                   // [S][5 * m]
  int *basis, *where;            // [S][m], [S][n + m + 1]
  double *x;                     // [S][n] out
  double *out;                   // [S][8] out: objective, status, pivots, phase-I pivots, refactorisations, Bland pivots
};
cudaError_t launch_lp(const LpLaunch &L, cudaStream_t st);

}  // namespace swb
