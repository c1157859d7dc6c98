/*
 * swb200.h — C-ABI of libswb200.so: the B200-native (sm_100a) replacement for the CPU solver calls
 * on Shockwave's per-round scheduling hot path.
 *
 * The reference (uw-mad-dash/shockwave) is pure Python; the arithmetic it delegates to
 * cvxpy -> Gurobi / ECOS is what these entry points replace.  Each entry point cites the reference
 * interface it stands in for.  Plain pointers and sizes only — no torch / pybind types.
 *
 * Conventions
 *   - every function returns an int status: 0 = ok, >0 = ok-with-note (see SWB_ST_*), <0 = error
 *     (SWB_ERR_*); swb_last_error() gives the text of the last error on the calling thread;
 *   - buffers are caller-owned; `*_dev` flags in the argument structs say whether the pointers are
 *     host (the default, e2e path: copies are done inside the call on the context's stream) or
 *     device pointers (inputs already resident in HBM);
 *   - one CUDA stream per context, no internal threads, not re-entrant per context (the reference
 *     calls the solver with Scheduler._scheduler_lock held: scheduler/scheduler.py:2188-2192).
 */
#ifndef SWB200_H
#define SWB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SWB_MAX_BASES 16
#define SWB_MAX_MODES 16

#define SWB_ST_OK 0
#define SWB_ST_FALLBACK 1 /* FTF rows infeasible -> relaxed objective + re-rank (shockwave.py:631-706) */

#define SWB_ERR_CUDA (-1)
#define SWB_ERR_ARG (-2)
#define SWB_ERR_NOMEM (-3)
#define SWB_ERR_STATE (-4)

typedef struct swb_ctx swb_ctx;

/* Scalars of one solve: the constructor kwargs of ShockwaveScheduler (scheduler/shockwave.py:21-86)
 * plus the per-call round pointer. */
typedef struct swb_params {
  int32_t ngpus;        /* G  : shockwave.py:40  */
  int32_t future_rounds;/* T  : shockwave.py:45  */
  int32_t round_ptr;    /* r  : shockwave.py:76  */
  int32_t nbases;       /* B  : len(logapx_bases), shockwave.py:60 */
  double round_duration;/* D  : shockwave.py:48  */
  double k;             /* shockwave.py:66  */
  double lam;           /* shockwave.py:85  */
  double rhomax;        /* shockwave.py:86  */
  double bases[SWB_MAX_BASES];   /* logapx_bases                      */
  double logv[SWB_MAX_BASES];    /* log(base) with log(0)->log(origin) : shockwave.py:339-347 */
} swb_params;

/* Result scalars of one solve (one per scenario). */
typedef struct swb_result {
  int32_t status;       /* SWB_ST_OK or SWB_ST_FALLBACK */
  int32_t m_evals;      /* makespan candidates evaluated */
  int32_t mu_iters;     /* price-bisection iterations in total */
  int32_t shortfall;    /* planned job-rounds the placement could not seat (0 = all seated) */
  int32_t placement;    /* fallback path: leading rounds seated by the priority round-sweep (the rest by the water-filling packer); 0 otherwise */
  int32_t flags;        /* bit 0: a gang width outside [1,255] was met in device-resident input (the call returns SWB_ERR_ARG) */
  double objective;     /* sum_j w_j plog_j/(J T) - k max_j rem_j of the RETURNED integral x */
  double welfare;       /* first term */
  double makespan;      /* max_j rem_j */
  double price;         /* clearing price mu (welfare per GPU-round) */
  double relaxed_objective; /* optimum of the continuous relaxation (n_j real) — upper bound */
} swb_result;

/* ---- context -------------------------------------------------------------------------------- */
int swb_create(swb_ctx **out, int device);
void swb_destroy(swb_ctx *ctx);
const char *swb_last_error(void);
int swb_version(void);
/* raw cudaStream_t of the context (so a host framework can order its own work after ours) */
void *swb_stream(swb_ctx *ctx);
int swb_sync(swb_ctx *ctx);

/* Options.  SWB_OPT_RELAXED_OPTIMUM: swb_solve / swb_round_solve additionally compute the EXACT optimum of
 * the continuous relaxation (x in [0,1]) into swb_result.relaxed_objective (about 10x slower; used by the
 * parity tests against the HiGHS LP relaxation).  Off: relaxed_objective holds the solver's own LP-style
 * upper estimate. */
#define SWB_OPT_RELAXED_OPTIMUM 1
/* SWB_OPT_SOLVE_CLUSTER: CTAs per scenario on the latency path of the market solve (8 = a thread-block cluster of 8
 * CTAs shares one scenario over distributed shared memory when few scenarios of >= 512 jobs are solved; 1 = always one
 * CTA per scenario).  The same setting lets the fallback re-rank search of the placement start from 8 seeds over a
 * cluster.  Per context.  Default 8. */
#define SWB_OPT_SOLVE_CLUSTER 2
/* Monte-Carlo (GBM) forecast inside swb_round_solve.  SWB_OPT_GBM_PATHS = P > 0: between the deterministic forecast
 * and the solve the remaining runtime of every job whose volatility model (swb_job_set_gbm) has drift or volatility
 * is replaced ON THE DEVICE by the mean of P geometric-Brownian-motion sample paths started at the deterministic
 * value (gbm.cu); jobs with mu = sigma = 0 keep the deterministic value bit for bit, so P > 0 with all-zero models
 * reproduces the reference's forecast exactly.  0 (default) = off.  SWB_OPT_GBM_SEED: stream seed;
 * SWB_OPT_GBM_HORIZON: horizon cap in epochs (default 256). */
/* SWB_OPT_RERANK_ITERS: budget (cancelled cycles per scenario) of the local search that follows the priority round-sweep
 * of the fallback re-rank (rank_in_schedule_jobs, shockwave.py:714-793); 0 = sweep only.  Default 400.  The search runs
 * when jobs x rounds^2 <= 256 Ki (e.g. 640 jobs at 20 rounds, 250 at 32); swb_result.flags >> 8 = cycles
 * cancelled (bits 8-19), >> 20 = which of the 8 starts of the multi-start search won (0 = the un-noised one; the search
 * runs 8 starts in a thread-block cluster when at most 18 scenarios of <= 4096 jobs are placed per call). */
#define SWB_OPT_RERANK_ITERS 6
/* SWB_OPT_RERANK_RESTARTS: rounds of perturb-and-continue (iterated local search) after the first local optimum of
 * every start; a round that does not improve is undone.  Default 2 (measured on the 128 recorded fallback solves of the
 * canonical run, profiles/rerank_restarts_r02.json: 0 rounds leave 3 solves above the reference's MIPGap of 1e-3, 1 round 1,
 * 2 rounds none, at +0.8 ms per round), at most 16, 0 = off. */
#define SWB_OPT_RERANK_RESTARTS 7
/* SWB_OPT_ASYNC_AUX: 1 = swb_gbm_forecast with device inputs AND device output, and swb_gbm_ensemble, return right after
 * their launches instead of synchronising the context's stream: a chain forecast -> ensemble -> swb_solve (device
 * pointers) then runs back to back on the device with ONE synchronisation, at the end of swb_solve.  The caller must
 * not read their outputs from another stream before a synchronising call (swb_sync, swb_solve, ...).  Default 0. */
#define SWB_OPT_ASYNC_AUX 8
#define SWB_OPT_GBM_PATHS 3
#define SWB_OPT_GBM_SEED 4
#define SWB_OPT_GBM_HORIZON 5
int swb_set_option(swb_ctx *ctx, int32_t option, int32_t value);

/* ---- the market solve on plain arrays ------------------------------------------------------- *
 * Replaces dynamic_eisenberg_gale_scheduling() (scheduler/shockwave.py:504-711) — model build +
 * Gurobi solve + infeasible->relaxed->re-rank fallback — and the rounding half of
 * construct_schedules() (shockwave.py:213-285).
 *
 * S independent scenarios are solved by one launch (one CTA each).  Per-job arrays are [S][J]
 * row-major when `per_scenario_jobs` != 0, else one shared [J] set; `prm` is [S].
 *   nworkers g_j (JobMetaData.py:57-60), epochs E_j (:62), epoch_progress c_j (:86),
 *   dbar_j = interpolate_epoch_duration (shockwave.py:322-324),
 *   rem_j  = dirichlet_posterior_remaining_runtime (JobMetaData.py:315-370),
 *   ftobj_j= finish_time_momentumed_average(share_series[j]) (shockwave.py:480-501),
 *   bfkey_j= back-fill sort key (remaining runtime at construct_schedules time, shockwave.py:261-267)
 * Outputs (caller-owned): x [S][J][T] uint8 (the rounded round-schedule variables),
 *   backfill [S][J][T] uint8 (1 where construct_schedules' work-conserving pass adds the job),
 *   nrounds [S][J] int32, weights [S][J] double (1 or the fallback priority), res [S].
 */
typedef struct swb_solve_args {
  int32_t S, J;
  int32_t per_scenario_jobs;
  int32_t on_device;            /* 0: all pointers are host memory; 1: all are device memory */
  const swb_params *prm;        /* [S], always HOST */
  const int32_t *g, *E, *c;
  const double *dbar, *rem, *ftobj, *bfkey;
  uint8_t *x, *backfill;        /* may be NULL */
  int32_t *nrounds;             /* may be NULL */
  double *weights;              /* may be NULL */
  swb_result *res;              /* [S], always HOST */
  /* optional packed outputs, [S][J][2] uint64 each: bit t of a job's 128-bit row = round t.  16 B per job
   * instead of T bytes — use these and leave x/backfill NULL when the device->host copy matters. */
  uint64_t *xmask, *bfmask;
} swb_solve_args;
int swb_solve(swb_ctx *ctx, const swb_solve_args *a);

/* ---- resident job table + dynamic-adaptation forecast ---------------------------------------- *
 * Replaces, per active job, JobMetaData.calibrate_profiled_epoch_duration (JobMetaData.py:225-288),
 * dirichlet_posterior_remaining_runtime (:315-370), interpolate_epoch_duration (shockwave.py:322-324)
 * and ShockwaveScheduler.finish_time_uniform_share (shockwave.py:88-120).
 * A job's static profile is uploaded once (add) into a device-resident table keyed by `slot`.
 */
int swb_job_add(swb_ctx *ctx, int32_t slot, int32_t nworkers, int32_t epochs, double epoch_nsamples,
                double timestamp_submit, const double *epoch_duration_preprofiled,
                const int32_t *bs_schedule);
int swb_job_remove(swb_ctx *ctx, int32_t slot);
/* Rows of the profile pools in use (high-water mark) and rows sitting in reusable holes: removed jobs give their
 * rows back, so `used_rows` tracks the LIVE jobs, not every job ever added.  Either pointer may be NULL. */
int swb_job_table_stats(swb_ctx *ctx, int64_t *used_rows, int64_t *hole_rows);
/* Volatility model of a resident job for the Monte-Carlo forecast: drift mu and volatility sigma per epoch of the
 * log epoch duration.  swb_job_add sets mu = 0 and sigma = the relative spread of the pre-profiled epoch durations
 * inside their batch-size modes (0 for the profiles the reference generates, utils.py:1350-1430). */
int swb_job_set_gbm(swb_ctx *ctx, int32_t slot, double mu, double sigma);

/* One full ShockwaveScheduler.round_schedule() re-solve (shockwave.py:122-166) for the jobs listed
 * in `slots` (metadata order).  Host inputs per job: epoch_progress, and the summary of the
 * throughput timeline (JobMetaData.py:235-249): measured sample count and last round (-1 = empty).
 * `gavel_round_duration` is JobMetaData.gavel_round_duration.  If `reestimate_share` the share
 * series of every job gets a new (round_ptr, finish-time-estimate) entry (shockwave.py:92-120).
 * `forecast_out` (may be NULL) receives 6 planes of [J] doubles: dbar, rem, ftobj, bfkey and the
 * fallback continuation rem_fb, bfkey_fb (used when res->status == SWB_ST_FALLBACK). */
typedef struct swb_round_args {
  int32_t J;
  int32_t reestimate_share;
  double gavel_round_duration;
  const int32_t *slots;         /* [J] host */
  const int32_t *epoch_progress;/* [J] host */
  const double *meas_nsamples;  /* [J] host */
  const int32_t *meas_end_round;/* [J] host, -1 when the timeline is empty */
  uint8_t *x, *backfill;        /* [J][T] host, out */
  int32_t *nrounds;             /* [J] host, out (may be NULL) */
  double *forecast_out;         /* [6][J] host, out (may be NULL) */
  swb_result *res;              /* host, out */
  /* optional packed outputs, [J][2] uint64 each (bit t of a job's 128-bit row = round t); x / backfill may then
   * be NULL: 16 B per job and matrix on the device->host copy instead of T bytes */
  uint64_t *xmask, *bfmask;
} swb_round_args;
int swb_round_solve(swb_ctx *ctx, const swb_params *prm, const swb_round_args *a);

/* Forecast only (same kernels as above, no solve); outputs [J] doubles each, host.  The share series
 * is advanced (when reestimate_share) but the calibration state is left untouched until
 * swb_forecast_commit() says which continuation the caller's solve took (fallback or not) and how
 * many times construct_schedules evaluated each job's sort key (ncal[j] = rounds with idle GPUs in
 * which job j was not scheduled; shockwave.py:254-267 -> JobMetaData.py:355,302). */
int swb_forecast(swb_ctx *ctx, const swb_params *prm, const swb_round_args *a, double *dbar,
                 double *rem, double *ftobj, double *bfkey, double *ft_estimate);
int swb_forecast_commit(swb_ctx *ctx, int32_t J, int32_t fallback, const int32_t *ncal);

/* ---- Gavel policies on a pooled (homogeneous) worker pool ------------------------------------- *
 * Replaces the cvxpy -> ECOS/Gurobi solve inside Policy.get_allocation() (scheduler/policies/*.py) when
 * every worker type that has capacity gives a job the same throughput (the non-Perf wrappers and
 * Shockwave's homogeneous clusters).  x[j] is the pooled time fraction; the caller splits it over the
 * worker types in proportion to their capacities.  Returns 0, or 1 when no feasible point was found.
 *   SWB_POL_MAXMIN   max_min_fairness.py:53-113    coef_j = thr_j * sf_j / (priority_j * proportional_thr_j)
 *   SWB_POL_FTF      finish_time_fairness.py:66-157 coef_j = thr_j, t = times_since_start,
 *                    n = num_steps_remaining, den_j = cumulative_isolated_time_j + n_j/isolated_thr_j
 *   SWB_POL_MTD      min_total_duration.py:55-135   coef_j = thr_j, n = num_steps_remaining
 *   SWB_POL_MAXSUM   max_sum_throughput.py:49-108   coef_j = thr_j / instance_cost; optional SLO floors in t:
 *                    t_j = num_steps_remaining_j / (SLO_j * thr_j) (0 = no SLO); returns 1 if the floors do not fit
 *   SWB_POL_ISOLATED isolated.py:35-55, proportional.py:26-43, gandiva_fair_proportional.py:26-41
 *                    coef_j = sf_j (Isolated) or 1 (Proportional / GandivaFair) */
#define SWB_POL_MAXMIN 1
#define SWB_POL_FTF 2
#define SWB_POL_MTD 3
#define SWB_POL_MAXSUM 4
#define SWB_POL_ISOLATED 5
int swb_policy_pooled(swb_ctx *ctx, int32_t mode, int32_t J, double N, const double *coef, const double *sf,
                      const double *t, const double *n, const double *den, double *x, double *objective);

/* ---- Gavel policies with heterogeneous worker types ------------------------------------------- *
 * Same programs as swb_policy_pooled (MAXMIN, FTF, MTD, MAXSUM with optional SLO floors) when the per-type throughputs of a
 * job differ — the general case of max_min_fairness.py:53-113, finish_time_fairness.py:66-157,
 * min_total_duration.py:55-135, max_sum_throughput.py:49-108 on a k80/p100/v100 cluster.  W <= 4 worker types (3 for MAXSUM),
 * each with N[w] > 0 workers (the caller drops empty types).  a is the J x W row-major matrix named per mode in
 * swb_policy_pooled (coef / throughput / throughput over cost); x is the J x W allocation (time fractions).
 * Solved exactly (bisection on the scalar objective, Dantzig-Wolfe on the W capacity rows with an exact master),
 * objective within 1e-12 relative of the LP optimum, every constraint certified.  MAXSUM accepts SLO floors
 * (max_sum_throughput.py:87-93): t[j] = needed throughput num_steps_remaining_j / SLO_j (0 = none) together with
 * den[w] = instance cost of worker type w (a = throughput / cost); returns 1 when the floors do not fit.  stats (optional, int32[2]):
 * pricing passes, feasibility checks.  Returns 0, or 1 when no feasible point was found. */
int swb_policy_hetero(swb_ctx *ctx, int32_t mode, int32_t J, int32_t W, const double *N, const double *a,
                      const double *sf, const double *t, const double *n, const double *den, double *x,
                      double *objective, int32_t *stats);

/* ---- water-filling max-min fairness: one iteration of WaterFillingAlgorithm ------------------------ *
 * Replaces the two solver calls inside the loop of _run_get_allocation_iterations
 * (scheduler/policies/max_min_fairness_water_filling.py:307-413):
 *   _get_allocation      :81-189   (cvxpy -> ECOS)     max c <= M :  net_j >= lower_j + c / mult_j  for mult_j > 0,
 *                                                       net_j >= lower_j otherwise,  net_j = thr_j.x_j / prop_j,
 *                                                       base constraints of policy.py:58-65
 *   _get_bottleneck_jobs :191-305  (cvxpy -> GLPK_MI)  max sum_j z_j :  every job keeps net_j >= so_far_j
 *                                                       (= lower_j + c / mult_j), z_j = 1 needs net_j >= so_far_j * slack
 * thr is the J x W throughput matrix (W <= 3 worker types, each with N[w] > 0), prop the proportional throughputs,
 * lower the normalised lower bounds (final value of a saturated job, so_far of the others), mult the reference's
 * multiplicative terms priority_j * scale_factor_j (0 for saturated / weightless jobs), M its big-M objective cap.
 * Out: x (J x W) = the LP's allocation, *c = its objective, z[J] = relaxed bottleneck indicator in [0, 1]
 * (the integer z of the reference rounds it; the caller treats z_j < 0.5 as "job j is a bottleneck").
 * Both programs run on the device (hetero.cu: bisection on the scalar, Dantzig-Wolfe on the coupling rows, every
 * feasibility claim certified).  stats (optional, int32[4]): pricing passes / feasibility checks of the two programs.
 * Returns 0, or 1 when the LP has no feasible point (x, c, z untouched). */
#define SWB_POL_WFILL 6
#define SWB_POL_WFZ 7
int swb_policy_waterfill_step(swb_ctx *ctx, int32_t J, int32_t W, const double *N, const double *thr, const double *sf,
                              const double *prop, const double *lower, const double *mult, double M, double slack,
                              double *x, double *c, double *z, int32_t *stats);

/* ---- Batch of sparse linear programs (the packing policies' LPs) ------------------------------ *
 * Replaces `cvxprob.solve(solver=self._solver)` in the *WithPacking policies
 * (scheduler/policies/max_min_fairness.py:317-410, finish_time_fairness.py:160-290, min_total_duration.py:138-234,
 *  max_sum_throughput.py:111-200; columns and rows from policy.py:68-193 `PolicyWithPacking`): one variable per
 * (job combination, worker type) — single jobs AND co-located pairs — so the per-job sub-problems the other policy
 * kernels decompose over are coupled and a general LP method is needed.
 *     maximise c'x   subject to   A x <= b,  x >= 0        (b may be negative; >= rows are passed negated)
 * S programs per call, one CTA each, sharing the CSC pattern (colp[n+1], rowi[nnz]) with per-program values
 * val[S][nnz], c[S][n], b[S][m].  Method: revised simplex with a dense fp64 basis inverse in HBM/L2 (rank-one
 * updates, Gauss-Jordan refactorisation every 96 pivots, Dantzig pricing with Bland's rule after 40 stalled
 * pivots, single-artificial phase I).  Exact to roundoff like the reference's solvers; optimal x is not unique.
 * Out: x[S][n], objective[S], status[S] (0 optimal, 1 infeasible, 2 unbounded, 3 pivot limit, 4 singular basis),
 * stats[S][4] (optional): pivots, phase-I pivots, refactorisations, Bland pivots.
 * Limits: m <= 2048, S <= 4096, S * m^2 * 16 B <= 8 GiB.  Returns 0, or SWB_ERR_STATE when any status >= 3. */
int swb_lp_solve(swb_ctx *ctx, int32_t S, int32_t m, int32_t n, int32_t nnz, const int32_t *colp, const int32_t *rowi,
                 const double *val, const double *c, const double *b, int32_t max_iter, double *x,
                 double *objective, int32_t *status, int32_t *stats);

/* ---- AlloX min-cost assignment --------------------------------------------------------------- *
 * Replaces scipy.optimize.linear_sum_assignment(q) in AlloXPolicy.get_allocation
 * (scheduler/policies/allox.py:108-144).  q is implicit: for job i and column col = k*n + j,
 *   q[i][col] = (k+1) * p[i][wtype[j]] + t[i],  p = num_steps_remaining / throughput, t = times_since_start,
 * m jobs, n workers (each with a type in [0, W)), m*n columns.  Output: the column assigned to every job
 * (worker = col % n, queue position = col / n) and the optimal total cost.  Exact (shortest augmenting
 * path, float64), like the reference's solver; optimal assignments are not unique. */
int swb_allox_assign(swb_ctx *ctx, int32_t m, int32_t n, int32_t W, const double *p, const double *t,
                     const int32_t *wtype, int32_t *col_of_job, double *total_cost);

/* ---- Gavel's per-round priority -> selection -> worker assignment ------------------------------------ *
 * Replaces, for single (unpacked) jobs, the step that follows get_allocation() in the reference's round loop:
 *   Scheduler._update_priorities, the "Compute priorities" half      scheduler/scheduler.py:3669-3724
 *   Scheduler._schedule_jobs_on_workers_helper, vanilla-Gavel branch scheduler/scheduler.py:1166-1258
 *   Scheduler._schedule_jobs_on_workers + _assign_workers_to_job     scheduler/scheduler.py:1306-1378, :1049-1110
 * Jobs are indexed in the iteration order of the reference's dicts (ties in its stable sorts resolve in that order).
 * Worker types: `W` types; per-(job, type) matrices are [J][W] indexed by the caller's type index; type_order lists
 * the type indices in PROCESSING order (the reference's possibly shuffled `worker_types`); nworkers / worker_ids are
 * given in that processing order (worker ids of a type in server order, servers concatenated).
 *   alloc      allocation[job][type], NaN when the job is not in the allocation (priority 0, not assigned)
 *   job_time   _job_time_so_far[job][type] (0 when absent); worker_time _worker_time_so_far[type]
 *   thr        throughput of the job on the type (only its sign / zero-ness is used)
 *   deficit    _deficits[type][job];  sf scale factors;  capacity cluster_spec[type]
 *   prev_type  type index of the job's assignment in the previous round (-1: none); prev_off [J+1] / prev_local: that
 *              assignment's workers as positions inside the type's worker list
 *   flags      bit 0: policy is Isolated_plus (the walk stops at the first job that does not fit), bit 1: FIFO
 * Outputs: prio [J][W]; n_sel [W] and sel_jobs [W][J] (per processing position, selection order);
 *   n_assigned, assign_job [J], assign_off [J+1], assign_workers: the new assignment in the reference's OrderedDict
 *   insertion order.  Returns 0, or SWB_ERR_STATE when the selected jobs do not fit the workers ("Could not assign
 *   workers to job", scheduler.py:1097-1100).  Bit-for-bit the dict code's result (integer / comparison work; the one
 *   division is the reference's own IEEE operation). */
typedef struct swb_gavel_round_args {
  int32_t J, W, flags;
  const int32_t *type_order, *capacity;
  const double *alloc, *job_time, *thr, *deficit;
  const double *worker_time;
  const int32_t *sf;
  const int32_t *nworkers, *worker_ids;
  const int32_t *prev_type, *prev_off, *prev_local;
  double *prio;
  int32_t *n_sel, *sel_jobs;
  int32_t *n_assigned, *assign_job, *assign_off, *assign_workers;
} swb_gavel_round_args;
int swb_gavel_round(swb_ctx *ctx, const swb_gavel_round_args *a);

/* ---- Monte-Carlo (geometric Brownian motion) throughput forecast -------------------------------- *
 * New capability, no reference counterpart (the reference's forecast is the deterministic
 * JobMetaData.dirichlet_posterior_remaining_runtime, JobMetaData.py:315-370, which this reduces to when
 * sigma = mu = 0).  For job j and LOCAL paths p in [0, P_local): global path id = path_offset + p,
 *   R = R0_j * mean_{h=1..H_j} exp((mu_j - sigma_j^2/2) h + sigma_j W_h).
 * out = [2][J] float64: sum_p R and sum_p R^2 (divide by the GLOBAL path count after the allreduce).
 * out_on_device bit 0: `out` is a device pointer (e.g. the tensor handed to ncclAllReduce); bit 1: R0, H, mu and sigma
 * are device pointers as well (inputs resident in HBM). */
int swb_gbm_forecast(swb_ctx *ctx, int32_t J, const double *R0, const int32_t *H, const double *mu,
                     const double *sigma, int64_t P_local, int64_t path_offset, uint64_t seed, double *out,
                     int32_t out_on_device);

/* Scenario ensemble from ONE Monte-Carlo forecast: rem_out[s][j] = max(0, mean_j + z[s] * std_j) with mean / std from
 * the (all-reduced) path sums — scenario s plans against the z[s]-sigma quantile of the remaining-runtime forecast.
 * sums_dev [2][J] and rem_out_dev [S][J] are DEVICE pointers, z [S] is host. */
int swb_gbm_ensemble(swb_ctx *ctx, int32_t S, int32_t J, double P_total, const double *sums_dev, const double *z,
                     double *rem_out_dev);

/* ---- dense market iteration over X[S][J][W][T] ------------------------------------------------ *
 * Primal-dual price-response iterations (preconditioned PDHG) on the dense allocation tensor (fp32, t innermost) of
 * the general volatile-Fisher-market relaxation: per-(job, type) progress rates, one capacity and one price per
 * (type, round).  Objective pieces as in scheduler/shockwave.py:565-568; base constraints as in
 * scheduler/policies/policy.py:58-65 applied per round.  `coarse_iters` iterations on the tensor coarsened to 4
 * super-rounds (prolongated afterwards; skipped when T < 16), then `iters` iterations of (dense pass + small dual
 * pass) on the full tensor; a dense pass reads X once and writes X once.  The returned X is feasible (a final pass
 * scales over-subscribed columns).  obj = [S][3]: relaxed objective, makespan and worst relative capacity violation
 * of the returned X.  dense_ms (may be NULL) = mean device time of the last (up to 16) full dense passes, one CUDA
 * event pair per pass. */
typedef struct swb_market_args {
  int32_t S, J, W, T;
  int32_t per_scenario_jobs;    /* job arrays are [S][J] (else shared [J]) */
  int32_t on_device;            /* g,E,c,dbar,rem,rate,X are device pointers */
  int32_t iters;                /* dense passes on the full tensor */
  int32_t coarse_iters;         /* passes on the time-coarsened tensor X_c[S][J][W][4], run first */
  int32_t warm_start;           /* 1: X holds the starting point, 0: start from X = 0 */
  float primal_weight;          /* PDHG step balance for the objective scaled by J T (tau = tau0/pw, sigma = sigma0 pw);
                                   0 = default (60; 1 with utility = 1) */
  int32_t utility;              /* 0: Shockwave's objective (PWL log + makespan term).  1: Eisenberg-Gale program
                                   max sum_j log(U_j), U_j = sum_wt rate_jw x_jwt over the jobs with E_j > 0 (E_j <= 0:
                                   job absent from the scenario) — the program of
                                   policies/max_min_fairness_strategy_proof.py:102-123 (geo_mean = the same argmax);
                                   c, dbar, rem and prm.k are ignored */
  const swb_params *prm;        /* [S] host: k, bases/logv, round_duration are used */
  const int32_t *g;
  const double *E, *c, *dbar, *rem;
  const float *rate;            /* [J][W] epochs of progress per round on worker type w */
  const double *Gw;             /* [W] host: workers per type (used when cap is NULL) */
  const double *cap;            /* [W][T] host: workers of type w available in round t; may be NULL */
  float *X;                     /* [S][J][W][T] in/out */
  double *obj;                  /* [S][3] host out, may be NULL */
  float *dense_ms;              /* host out, may be NULL */
} swb_market_args;
int swb_market_pgd(swb_ctx *ctx, const swb_market_args *a);

/* ---- simulator round loop on the device (SURVEY §8(f)-4) ---------------------------------------- *
 * The round loop of `Scheduler.simulate()` (scheduler/scheduler.py:1878-2250: jump to the next event, book the progress
 * of the jobs that ran, retire finished jobs, admit arrivals) with the pieces of `_get_job_steps_and_finish_times`
 * (:1467-1512), `_get_num_steps` (:1425-1465), `_done_callback` (:4341-4700), `_update_throughput` (:549-571),
 * `_remove_job` (:808-830) and `_update_shockwave_scheduler` (:2270-2342) that act on STATIC jobs of a trace on one
 * worker type — for S what-if scenarios of the same trace at once, one CTA per scenario, state resident in HBM.
 * The policy stays outside: every step takes the jobs chosen for the round (chosen[S][J], 1 = run) — from
 * ShockwaveScheduler.round_schedule(), a Gavel policy + swb_gavel_round, or a recorded schedule (swb_sim_replay runs
 * ALL rounds in one launch, no host in the loop).  Arithmetic = the reference's, in its order (IEEE double / int64):
 * completion times, makespan and measured throughputs are bit-identical to the reference loop on the same schedule
 * (tests/test_oracle_sim_loop.py, tests/test_gpu_sim.py).  Dynamic adaptation — accordion / gns batch-size rescaling,
 * `_simulate_accordion` :1658-1727, `_simulate_gns` :1604-1656, `_scale_bs_and_iters` :4731-4935 — runs from tables
 * (swb_sim_set_dynamic); the micro-task failure branch of `_done_callback` (:4497-4570, five empty rounds in a row drop
 * the job) is part of the loop.  Several worker types (static jobs): swb_sim_set_worker_types.  Not covered: job pairs
 * (packing), the `ideal` mode. */
typedef struct swb_sim swb_sim;
typedef struct swb_sim_trace {
  int32_t J;
  int32_t reserved;
  const double *arrival;          /* [J] non-decreasing (scheduler.py:1842-1843) */
  const int64_t *total_steps;     /* [J] job.total_steps */
  const int32_t *scale_factor;    /* [J] gang width */
  const double *throughput;       /* [J] steps/s of the job on the worker type (oracle throughputs, "null" co-location) */
  const double *duration;         /* [J] job.duration (over-deadline rule: run time > int(1.5 duration)) */
  const int32_t *batch_size;      /* [J] */
  const int64_t *dataset_len;     /* [J] samples per epoch (scheduler.py:73-81 dataset_size_dict) */
  const int32_t *adaptation_mode; /* [J] or NULL: 0 static, 1 accordion, 2 gns; a trace with non-static jobs needs
                                     swb_sim_set_dynamic before the first round */
} swb_sim_trace;
/* Tables of the dynamic-adaptation jobs; batch_size / total_steps / throughput of the trace are the ORIGINAL values.
 * shockwave_b200/simulate.py::build_dynamic_tables lays them out from the reference's rules (INTEGRATION.md). */
typedef struct swb_sim_dynamic {
  const int32_t *mode;        /* [J] 0 static, 1 accordion, 2 gns */
  const int32_t *bs_max;      /* [J] batch size at which no scale-up is requested (scheduler.py:1636-1646, :1699-1709) */
  const int32_t *bs_min;      /* [J] batch size at which no scale-down is requested (:1711-1721) */
  const int32_t *bs_big;      /* [J] accordion's scale-up target max_bs_dict[model] (:4756-4761); <= 0: none */
  const int32_t *orig_locked; /* [J] 1: the original batch size is max_bs_dict[model]: every request is dropped (:4767-4775) */
  const int32_t *acc_skip;    /* [J] 1: accordion never applies (Transformer, :1667-1669) */
  const int64_t *pat_off;     /* [J+1] offsets into pattern */
  const int32_t *pattern;     /* accordion: 1 = critical regime at that epoch (:1670-1692); gns: batch size at that epoch
                                 (utils.get_gns_bs_pattern with >= 762 epochs; the loop applies the reference's
                                 "last entry is never scaled" rule for epochs >= 758 itself) */
  int32_t n_levels;           /* K <= 8 */
  int32_t reserved;
  const int32_t *lvl_bs;      /* [J][K] batch sizes the job can move to (0 = unused) */
  const double *lvl_thr;      /* [J][K] throughput of the job at that batch size (<= 0: not in the throughput file) */
} swb_sim_dynamic;
int swb_sim_set_dynamic(swb_sim *sim, const swb_sim_dynamic *tables);
/* Several worker types (the heterogeneity-aware Gavel policies on mixed clusters): per-type throughputs
 * throughput[J][W] (`Scheduler._throughputs[job][worker_type]`, read by `_get_job_steps_and_finish_times`
 * scheduler.py:1467-1512; 0 = the job cannot run on that type) and worker counts ngpus[W], W <= 8.  Afterwards
 * chosen[s][j] = 1 + index of the type job j runs on in the round (0 = not chosen), capacity is checked per type, and the
 * `throughput` / `ngpus` of swb_sim_create are not used.  Static jobs only (the reference's batch-size rescale keeps its
 * progress counters on v100 alone, :4896-4925): refused for a trace with adaptation modes, and swb_sim_set_dynamic is
 * refused afterwards.  Call before swb_sim_begin. */
int swb_sim_set_worker_types(swb_sim *sim, int32_t W, const double *throughput, const int32_t *ngpus);
typedef struct swb_sim_scn {      /* per scenario, after a step */
  double now;                     /* Scheduler._current_timestamp; at the end of the run: the makespan */
  double round_start, round_end;  /* current_round_start_time / _end_time (NaN = None) */
  int32_t rounds;                 /* completed rounds (_num_completed_rounds) */
  int32_t remaining;              /* jobs of the trace not completed yet */
  int32_t n_active;               /* live jobs (len(self._jobs)) */
  int32_t done;                   /* 1: the reference's loop has left (all jobs completed, or no live job) */
  int32_t err;                    /* bit 0: chosen gangs exceed ngpus; bit 1: nothing running and no arrival left
                                     (the reference raises); bit 2: a job's epoch left its dynamic-adaptation table;
                                     bit 3: a job was chosen on a worker type where its throughput is 0 (the reference
                                     raises, scheduler.py:1494-1504) */
  int32_t reserved;
} swb_sim_scn;
int swb_sim_create(int32_t device, const swb_sim_trace *trace, int32_t S, int32_t ngpus, double time_per_iteration,
                   double round_duration, swb_sim **out);
void swb_sim_destroy(swb_sim *sim);
/* iteration 0: timestamp = first arrival, admit the jobs that have arrived.  status[S][J] (may be NULL): 0 queued,
 * 1 live, 2 completed. */
int swb_sim_begin(swb_sim *sim, swb_sim_scn *scn, uint8_t *status);
/* run one round with chosen[S][J] (host) and advance to the next decision point.  Outputs (host, any may be NULL):
 * scn[S]; status[S][J]; epoch[S][J] = epoch progress of the jobs that ran (-1: the job completed; untouched otherwise);
 * tl_ns[S][J], tl_end[S][J] = measured-samples sum and last measured round of the throughput timeline
 * (JobMetaData.py:235-249) — what ShockwaveScheduler's forecast takes per job. */
int swb_sim_step(swb_sim *sim, const uint8_t *chosen, swb_sim_scn *scn, uint8_t *status, int32_t *epoch, double *tl_ns,
                 int32_t *tl_end);
/* begin + R rounds in ONE launch from a known schedule: schedule[R][J] shared by the scenarios (per_scenario = 0) or
 * schedule[R][S][J]; scenarios that finish earlier ignore the rest. */
int swb_sim_replay(swb_sim *sim, const uint8_t *schedule, int32_t R, int32_t per_scenario, swb_sim_scn *scn);
/* per-job results [S][J] (host, any may be NULL): completion time - arrival (NaN: not completed), steps run, cumulative
 * run time, throughput measured in the job's latest round. */
int swb_sim_results(swb_sim *sim, double *jct, int64_t *steps_run, double *run_time, double *measured_throughput);
/* what the Gavel mechanism between two rounds reads of every job [S][J] (host, any may be NULL): current total steps /
 * throughput / batch size (they change with a rescale), execution time booked for the job's latest round and its finish
 * time (`_job_time_so_far`, `_worker_time_so_far` accounting of `_done_callback`, scheduler.py:4660-4672, in completion
 * order), failed attempts in a row (> 0: the latest round was a micro-task failure), ran = 1 for the jobs of that round. */
int swb_sim_job_state(swb_sim *sim, int64_t *total_steps, double *throughput, int32_t *batch_size, double *exec_time,
                      double *finish_time, uint8_t *failed_attempts, uint8_t *ran);

/* Device time (CUDA events on the context's stream) of the two kernels of the latest solve pass and
 * the number of solve+place passes that call took (1 + packing-feedback re-solves). */
int swb_last_timings(swb_ctx *ctx, double *ms_solve, double *ms_place, int32_t *passes);

#ifdef __cplusplus
}
#endif
#endif /* SWB200_H */
