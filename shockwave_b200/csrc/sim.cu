// swb_sim_*: the reference simulator's round loop for S what-if scenarios of one static trace, on the device
// (sim_core.cuh; SURVEY §8(f)-4).  One CTA per scenario; a launch runs R rounds back to back (R = 1 when a policy on the
// host / another kernel chooses the jobs of every round, R = all rounds when the schedule is known: replay).
#include <math.h>
#include <new>
#include <string.h>
#include <string>
#include <vector>

#include "swb_internal.h"
#include "sim_core.cuh"

#define SIM_THREADS 256

namespace swb {

struct SimLaunch {
  sim::Trace T;
  sim::State X;            // [S][J] bases
  sim::Scn *scn;           // [S]
  const unsigned char *chosen;
  long long stride_r, stride_s;   // chosen[r * stride_r + s * stride_s + j]
  int R, begin, ngpus;
  double tpi, grd;
};

__global__ void __launch_bounds__(SIM_THREADS) sim_kernel(SimLaunch L) {
  __shared__ double sd[SIM_THREADS];
  __shared__ long long si[SIM_THREADS];
  const size_t o = (size_t)blockIdx.x * L.T.J;
  sim::State X = L.X;
  X.status += o; X.ranprev += o; X.steps_run += o; X.nsteps += o; X.run_time += o; X.latest += o; X.jct += o;
  X.fin += o; X.tl_ns += o; X.thr_meas += o; X.tl_prev += o; X.tl_end += o; X.epoch += o;
  X.running += o; X.flag += o; X.fails += o; X.cbs += o; X.ctotal += o; X.cspe += o; X.cthr += o; X.last_ex += o;
  sim::Shared sh{sd, si};
  sim::Scn *scn = L.scn + blockIdx.x;
  if (L.begin) sim::scenario_begin(L.T, X, scn, sh);
  for (int r = 0; r < L.R; ++r)
    sim::scenario_step(L.T, X, scn, L.chosen + (size_t)r * L.stride_r + (size_t)blockIdx.x * L.stride_s, L.ngpus, L.tpi,
                       L.grd, sh);
}

}  // namespace swb

struct swb_sim {
  int device = 0, S = 0, J = 0, ngpus = 0, begun = 0;
  double tpi = 0, grd = 0;
  cudaStream_t st = nullptr;
  DBuf arena;                   // trace + state, one allocation
  DBuf dyn_arena;               // tables of swb_sim_set_dynamic
  DBuf wt_arena;                // tables of swb_sim_set_worker_types
  int needs_dynamic = 0;        // the trace names non-static jobs: tables are required before the first round
  DBuf d_chosen;                // chosen / schedule of the latest step or replay
  PinBuf h_pin;                 // pinned staging of the per-step outputs
  swb::sim::Trace T;
  swb::sim::State X;
  swb::sim::Scn *scn = nullptr;
};

static size_t al(size_t b) { return (b + 255) & ~(size_t)255; }

extern "C" {

void swb_sim_destroy(swb_sim *m) {
  if (!m) return;
  cudaSetDevice(m->device);
  if (m->st) cudaStreamSynchronize(m->st);
  if (m->st) cudaStreamDestroy(m->st);
  delete m;      // the buffers free themselves
}

int swb_sim_create(int32_t device, const swb_sim_trace *tr, int32_t S, int32_t ngpus, double time_per_iteration,
                   double round_duration, swb_sim **out) {
  if (!tr || !out) return swb_set_error(SWB_ERR_ARG, "swb_sim_create: null argument");
  *out = nullptr;
  const int J = tr->J;
  if (J <= 0 || J > (1 << 20) || S <= 0 || S > 65535 || ngpus <= 0 || !(time_per_iteration > 0) || !(round_duration > 0))
    return swb_set_error(SWB_ERR_ARG, "swb_sim_create: need 1 <= J <= 2^20, 1 <= S <= 65535, ngpus > 0, durations > 0");
  if (!tr->arrival || !tr->total_steps || !tr->scale_factor || !tr->throughput || !tr->duration || !tr->batch_size ||
      !tr->dataset_len)
    return swb_set_error(SWB_ERR_ARG, "swb_sim_create: null trace array");
  std::vector<double> dur15(J);
  std::vector<long long> spe(J);
  int any_dynamic = 0;
  for (int j = 0; j < J; ++j) {
    if (j && tr->arrival[j] < tr->arrival[j - 1])
      return swb_set_error(SWB_ERR_ARG, "swb_sim_create: arrival times must be non-decreasing (scheduler.py:1842-1843)");
    if (!(tr->throughput[j] > 0) || tr->total_steps[j] <= 0 || tr->scale_factor[j] <= 0 || tr->batch_size[j] <= 0 ||
        tr->dataset_len[j] <= 0 || !(tr->duration[j] >= 0) || !(tr->arrival[j] >= 0))
      return swb_set_error(SWB_ERR_ARG, "swb_sim_create: throughput, total_steps, scale_factor, batch_size, dataset_len "
                                        "must be positive, duration / arrival non-negative");
    if (tr->adaptation_mode && (tr->adaptation_mode[j] < 0 || tr->adaptation_mode[j] > 2))
      return swb_set_error(SWB_ERR_ARG, "swb_sim_create: adaptation_mode must be 0 (static), 1 (accordion) or 2 (gns)");
    if (tr->adaptation_mode && tr->adaptation_mode[j] != 0) any_dynamic = 1;
    dur15[j] = (double)(long long)(tr->duration[j] * 1.5);
    spe[j] = (tr->dataset_len[j] + tr->batch_size[j] - 1) / tr->batch_size[j];
  }
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0)
    return swb_set_error(SWB_ERR_CUDA, "swb_sim_create: no CUDA device (this library has no CPU path)");
  if (device < 0 || device >= ndev) return swb_set_error(SWB_ERR_ARG, "swb_sim_create: bad device index");
  swb_sim *m = new (std::nothrow) swb_sim;
  if (!m) return swb_set_error(SWB_ERR_CUDA, "swb_sim_create: out of memory");
  m->needs_dynamic = any_dynamic;
  m->device = device; m->S = S; m->J = J; m->ngpus = ngpus; m->tpi = time_per_iteration; m->grd = round_duration;
  cudaError_t e = cudaSetDevice(device);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&m->st, cudaStreamNonBlocking);
  const size_t sj = (size_t)S * J;
  // arena: trace [J] (5 x 8 B + 2 x 4 B), state [S][J], scenario scalars [S]
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off += al(bytes); return o; };
  const size_t o_arr = take((size_t)J * 8), o_tot = take((size_t)J * 8), o_thr = take((size_t)J * 8),
               o_d15 = take((size_t)J * 8), o_spe = take((size_t)J * 8), o_ds = take((size_t)J * 8), o_sf = take((size_t)J * 4),
               o_bs = take((size_t)J * 4);
  const size_t o_status = take(sj), o_ranprev = take(sj), o_steps = take(sj * 8), o_nsteps = take(sj * 8),
               o_rt = take(sj * 8), o_latest = take(sj * 8), o_jct = take(sj * 8), o_fin = take(sj * 8),
               o_tlns = take(sj * 8), o_tm = take(sj * 8), o_tlprev = take(sj * 4), o_tlend = take(sj * 4),
               o_epoch = take(sj * 4), o_running = take(sj), o_flag = take(sj), o_fails = take(sj), o_cbs = take(sj * 4),
               o_ctotal = take(sj * 8), o_cspe = take(sj * 8), o_cthr = take(sj * 8), o_lastex = take(sj * 8),
               o_scn = take((size_t)S * sizeof(swb::sim::Scn));
  if (e == cudaSuccess) e = m->arena.need(off, m->st);
  if (e != cudaSuccess) {
    swb_sim_destroy(m);
    return swb_set_error(SWB_ERR_CUDA, (std::string("swb_sim_create: ") + cudaGetErrorString(e)).c_str());
  }
  char *b = m->arena.as<char>();
  auto up = [&](size_t o, const void *src, size_t bytes) {
    return cudaMemcpyAsync(b + o, src, bytes, cudaMemcpyHostToDevice, m->st);
  };
  e = up(o_arr, tr->arrival, (size_t)J * 8);
  if (e == cudaSuccess) e = up(o_tot, tr->total_steps, (size_t)J * 8);
  if (e == cudaSuccess) e = up(o_thr, tr->throughput, (size_t)J * 8);
  if (e == cudaSuccess) e = up(o_d15, dur15.data(), (size_t)J * 8);
  if (e == cudaSuccess) e = up(o_spe, spe.data(), (size_t)J * 8);
  if (e == cudaSuccess) e = up(o_ds, tr->dataset_len, (size_t)J * 8);
  if (e == cudaSuccess) e = up(o_sf, tr->scale_factor, (size_t)J * 4);
  if (e == cudaSuccess) e = up(o_bs, tr->batch_size, (size_t)J * 4);
  if (e == cudaSuccess) e = cudaStreamSynchronize(m->st);      // dur15 / spe are locals
  if (e != cudaSuccess) {
    swb_sim_destroy(m);
    return swb_set_error(SWB_ERR_CUDA, (std::string("swb_sim_create: ") + cudaGetErrorString(e)).c_str());
  }
  m->T = swb::sim::Trace{};
  m->T.J = J; m->T.arrival = (const double *)(b + o_arr); m->T.total = (const long long *)(b + o_tot);
  m->T.sf = (const int *)(b + o_sf); m->T.thr = (const double *)(b + o_thr); m->T.dur15 = (const double *)(b + o_d15);
  m->T.bs = (const int *)(b + o_bs); m->T.spe = (const long long *)(b + o_spe); m->T.ds = (const long long *)(b + o_ds);
  m->X.status = (unsigned char *)(b + o_status); m->X.ranprev = (unsigned char *)(b + o_ranprev);
  m->X.steps_run = (long long *)(b + o_steps); m->X.nsteps = (long long *)(b + o_nsteps);
  m->X.run_time = (double *)(b + o_rt); m->X.latest = (double *)(b + o_latest); m->X.jct = (double *)(b + o_jct);
  m->X.fin = (double *)(b + o_fin); m->X.tl_ns = (double *)(b + o_tlns); m->X.thr_meas = (double *)(b + o_tm);
  m->X.tl_prev = (int *)(b + o_tlprev); m->X.tl_end = (int *)(b + o_tlend); m->X.epoch = (int *)(b + o_epoch);
  m->X.running = (unsigned char *)(b + o_running); m->X.flag = (unsigned char *)(b + o_flag);
  m->X.fails = (unsigned char *)(b + o_fails); m->X.cbs = (int *)(b + o_cbs); m->X.ctotal = (long long *)(b + o_ctotal);
  m->X.cspe = (long long *)(b + o_cspe); m->X.cthr = (double *)(b + o_cthr); m->X.last_ex = (double *)(b + o_lastex);
  m->scn = (swb::sim::Scn *)(b + o_scn);
  *out = m;
  return 0;
}

// shared tail of begin / step / replay: launch, bring the requested per-step views back through pinned memory
static int sim_run(swb_sim *m, const unsigned char *d_chosen, long long stride_r, long long stride_s, int R, int begin,
                   swb_sim_scn *scn, uint8_t *status, int32_t *epoch, double *tl_ns, int32_t *tl_end) {
  swb::SimLaunch L;
  L.T = m->T; L.X = m->X; L.scn = m->scn; L.chosen = d_chosen; L.stride_r = stride_r; L.stride_s = stride_s;
  L.R = R; L.begin = begin; L.ngpus = m->ngpus; L.tpi = m->tpi; L.grd = m->grd;
  // block size: a multiple of 32 (the reductions shuffle over full warps), one job per thread up to 256
  const int threads = m->J <= 32 ? 32 : m->J <= 64 ? 64 : m->J <= 128 ? 128 : SIM_THREADS;
  swb::sim_kernel<<<m->S, threads, 0, m->st>>>(L);
  CK(cudaGetLastError());
  const size_t sj = (size_t)m->S * m->J;
  CK(m->h_pin.need(al((size_t)m->S * sizeof(swb_sim_scn)) + al(sj) + 2 * al(sj * 4) + al(sj * 8)));
  unsigned char *p = m->h_pin.as<unsigned char>();
  unsigned char *p_scn = p; p += al((size_t)m->S * sizeof(swb_sim_scn));
  unsigned char *p_st = p; p += al(sj);
  unsigned char *p_ep = p; p += al(sj * 4);
  unsigned char *p_te = p; p += al(sj * 4);
  unsigned char *p_ns = p;
  if (scn) CK(cudaMemcpyAsync(p_scn, m->scn, (size_t)m->S * sizeof(swb_sim_scn), cudaMemcpyDeviceToHost, m->st));
  if (status) CK(cudaMemcpyAsync(p_st, m->X.status, sj, cudaMemcpyDeviceToHost, m->st));
  if (epoch) CK(cudaMemcpyAsync(p_ep, m->X.epoch, sj * 4, cudaMemcpyDeviceToHost, m->st));
  if (tl_end) CK(cudaMemcpyAsync(p_te, m->X.tl_end, sj * 4, cudaMemcpyDeviceToHost, m->st));
  if (tl_ns) CK(cudaMemcpyAsync(p_ns, m->X.tl_ns, sj * 8, cudaMemcpyDeviceToHost, m->st));
  CK(cudaStreamSynchronize(m->st));
  if (scn) memcpy(scn, p_scn, (size_t)m->S * sizeof(swb_sim_scn));
  if (status) memcpy(status, p_st, sj);
  if (epoch) memcpy(epoch, p_ep, sj * 4);
  if (tl_end) memcpy(tl_end, p_te, sj * 4);
  if (tl_ns) memcpy(tl_ns, p_ns, sj * 8);
  return 0;
}

int swb_sim_set_dynamic(swb_sim *m, const swb_sim_dynamic *d) {
  if (!m || !d) return swb_set_error(SWB_ERR_ARG, "swb_sim_set_dynamic: null argument");
  if (!d->mode || !d->bs_max || !d->bs_min || !d->bs_big || !d->orig_locked || !d->acc_skip || !d->pat_off || !d->lvl_bs ||
      !d->lvl_thr)
    return swb_set_error(SWB_ERR_ARG, "swb_sim_set_dynamic: null table");
  if (m->T.thr_w) return swb_set_error(SWB_ERR_ARG, "swb_sim_set_dynamic: several worker types run static jobs only");
  const int J = m->J, K = d->n_levels;
  if (K <= 0 || K > SIM_MAX_LEVELS) return swb_set_error(SWB_ERR_ARG, "swb_sim_set_dynamic: n_levels must be in [1, 8]");
  if (d->pat_off[0] != 0) return swb_set_error(SWB_ERR_ARG, "swb_sim_set_dynamic: pat_off[0] must be 0");
  for (int j = 0; j < J; ++j) {
    if (d->pat_off[j + 1] < d->pat_off[j]) return swb_set_error(SWB_ERR_ARG, "swb_sim_set_dynamic: pat_off must be non-decreasing");
    if (d->mode[j] < 0 || d->mode[j] > 2) return swb_set_error(SWB_ERR_ARG, "swb_sim_set_dynamic: mode must be 0, 1 or 2");
    if (d->mode[j] == 2 && d->pat_off[j + 1] - d->pat_off[j] < 762)
      return swb_set_error(SWB_ERR_ARG, "swb_sim_set_dynamic: a gns job needs a pattern of >= 762 epochs (scheduler.py:1617-1622)");
  }
  const long long np = d->pat_off[J];
  if (np > 0 && !d->pattern) return swb_set_error(SWB_ERR_ARG, "swb_sim_set_dynamic: null pattern");
  CK(cudaSetDevice(m->device));
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off += al(bytes ? bytes : 1); return o; };
  const size_t o_mode = take((size_t)J * 4), o_max = take((size_t)J * 4), o_min = take((size_t)J * 4), o_big = take((size_t)J * 4),
               o_lock = take((size_t)J * 4), o_skip = take((size_t)J * 4), o_off = take((size_t)(J + 1) * 8),
               o_pat = take((size_t)np * 4), o_lb = take((size_t)J * K * 4), o_lt = take((size_t)J * K * 8);
  CK(cudaStreamSynchronize(m->st));      // a launched round may still read the old tables
  CK(m->dyn_arena.need(off, m->st));
  char *b = m->dyn_arena.as<char>();
  auto up = [&](size_t o, const void *src, size_t bytes) {
    return bytes ? cudaMemcpyAsync(b + o, src, bytes, cudaMemcpyHostToDevice, m->st) : cudaSuccess;
  };
  CK(up(o_mode, d->mode, (size_t)J * 4)); CK(up(o_max, d->bs_max, (size_t)J * 4)); CK(up(o_min, d->bs_min, (size_t)J * 4));
  CK(up(o_big, d->bs_big, (size_t)J * 4)); CK(up(o_lock, d->orig_locked, (size_t)J * 4));
  CK(up(o_skip, d->acc_skip, (size_t)J * 4)); CK(up(o_off, d->pat_off, (size_t)(J + 1) * 8));
  CK(up(o_pat, d->pattern, (size_t)np * 4)); CK(up(o_lb, d->lvl_bs, (size_t)J * K * 4));
  CK(up(o_lt, d->lvl_thr, (size_t)J * K * 8));
  CK(cudaStreamSynchronize(m->st));
  m->T.mode = (const int *)(b + o_mode); m->T.bs_max = (const int *)(b + o_max); m->T.bs_min = (const int *)(b + o_min);
  m->T.bs_big = (const int *)(b + o_big); m->T.orig_locked = (const int *)(b + o_lock); m->T.acc_skip = (const int *)(b + o_skip);
  m->T.pat_off = (const long long *)(b + o_off); m->T.pattern = (const int *)(b + o_pat); m->T.K = K;
  m->T.lvl_bs = (const int *)(b + o_lb); m->T.lvl_thr = (const double *)(b + o_lt);
  m->needs_dynamic = 0;
  return 0;
}

int swb_sim_set_worker_types(swb_sim *m, int32_t W, const double *throughput, const int32_t *ngpus) {
  if (!m || !throughput || !ngpus) return swb_set_error(SWB_ERR_ARG, "swb_sim_set_worker_types: null argument");
  if (W < 1 || W > SIM_MAX_TYPES) return swb_set_error(SWB_ERR_ARG, "swb_sim_set_worker_types: need 1 <= W <= 8");
  if (m->needs_dynamic || m->T.mode)
    return swb_set_error(SWB_ERR_ARG, "swb_sim_set_worker_types: several worker types run static jobs only (the reference "
                                      "rescales a job's progress on v100 alone, scheduler.py:4896-4925)");
  const int J = m->J;
  for (int w = 0; w < W; ++w)
    if (ngpus[w] < 0) return swb_set_error(SWB_ERR_ARG, "swb_sim_set_worker_types: negative worker count");
  for (size_t i = 0; i < (size_t)J * W; ++i)
    if (!(throughput[i] >= 0.0)) return swb_set_error(SWB_ERR_ARG, "swb_sim_set_worker_types: throughput must be >= 0 (0 = the job cannot run on that type)");
  CK(cudaSetDevice(m->device));
  const size_t o_thr = 0, o_cap = al((size_t)J * W * 8), total = o_cap + al((size_t)W * 4);
  CK(cudaStreamSynchronize(m->st));      // a launched round may still read the old tables
  m->T.thr_w = nullptr; m->T.cap_w = nullptr; m->T.W = 0;
  CK(m->wt_arena.need(total, m->st));
  char *b = m->wt_arena.as<char>();
  CK(cudaMemcpyAsync(b + o_thr, throughput, (size_t)J * W * 8, cudaMemcpyHostToDevice, m->st));
  CK(cudaMemcpyAsync(b + o_cap, ngpus, (size_t)W * 4, cudaMemcpyHostToDevice, m->st));
  CK(cudaStreamSynchronize(m->st));
  m->T.W = W; m->T.thr_w = (const double *)(b + o_thr); m->T.cap_w = (const int *)(b + o_cap);
  return 0;
}

int swb_sim_begin(swb_sim *m, swb_sim_scn *scn, uint8_t *status) {
  if (!m) return swb_set_error(SWB_ERR_ARG, "swb_sim_begin: null handle");
  if (m->needs_dynamic)
    return swb_set_error(SWB_ERR_STATE, "swb_sim_begin: the trace has accordion / gns jobs: call swb_sim_set_dynamic first");
  CK(cudaSetDevice(m->device));
  m->begun = 1;
  return sim_run(m, nullptr, 0, 0, 0, 1, scn, status, nullptr, nullptr, nullptr);
}

int swb_sim_step(swb_sim *m, const uint8_t *chosen, swb_sim_scn *scn, uint8_t *status, int32_t *epoch, double *tl_ns,
                 int32_t *tl_end) {
  if (!m || !chosen) return swb_set_error(SWB_ERR_ARG, "swb_sim_step: null argument");
  if (!m->begun) return swb_set_error(SWB_ERR_STATE, "swb_sim_step: call swb_sim_begin first");
  CK(cudaSetDevice(m->device));
  const size_t sj = (size_t)m->S * m->J;
  CK(m->d_chosen.upload(chosen, sj, m->st));
  return sim_run(m, m->d_chosen.as<unsigned char>(), 0, m->J, 1, 0, scn, status, epoch, tl_ns, tl_end);
}

int swb_sim_replay(swb_sim *m, const uint8_t *schedule, int32_t R, int32_t per_scenario, swb_sim_scn *scn) {
  if (!m || !schedule || R <= 0) return swb_set_error(SWB_ERR_ARG, "swb_sim_replay: null argument or R <= 0");
  CK(cudaSetDevice(m->device));
  const size_t per_round = per_scenario ? (size_t)m->S * m->J : (size_t)m->J;
  if (per_round * (size_t)R > ((size_t)4 << 30)) return swb_set_error(SWB_ERR_ARG, "swb_sim_replay: schedule above 4 GiB");
  if (m->needs_dynamic)
    return swb_set_error(SWB_ERR_STATE, "swb_sim_replay: the trace has accordion / gns jobs: call swb_sim_set_dynamic first");
  CK(m->d_chosen.upload(schedule, per_round * (size_t)R, m->st));
  m->begun = 1;
  return sim_run(m, m->d_chosen.as<unsigned char>(), (long long)per_round, per_scenario ? m->J : 0, R, 1, scn, nullptr, nullptr, nullptr, nullptr);
}

int swb_sim_results(swb_sim *m, double *jct, int64_t *steps_run, double *run_time, double *measured_throughput) {
  if (!m) return swb_set_error(SWB_ERR_ARG, "swb_sim_results: null handle");
  CK(cudaSetDevice(m->device));
  const size_t sj = (size_t)m->S * m->J;
  if (jct) CK(cudaMemcpyAsync(jct, m->X.jct, sj * 8, cudaMemcpyDeviceToHost, m->st));
  if (steps_run) CK(cudaMemcpyAsync(steps_run, m->X.steps_run, sj * 8, cudaMemcpyDeviceToHost, m->st));
  if (run_time) CK(cudaMemcpyAsync(run_time, m->X.run_time, sj * 8, cudaMemcpyDeviceToHost, m->st));
  if (measured_throughput) CK(cudaMemcpyAsync(measured_throughput, m->X.thr_meas, sj * 8, cudaMemcpyDeviceToHost, m->st));
  CK(cudaStreamSynchronize(m->st));
  return 0;
}

int swb_sim_job_state(swb_sim *m, int64_t *total_steps, double *throughput, int32_t *batch_size, double *exec_time,
                      double *finish_time, uint8_t *failed_attempts, uint8_t *ran) {
  if (!m) return swb_set_error(SWB_ERR_ARG, "swb_sim_job_state: null handle");
  CK(cudaSetDevice(m->device));
  const size_t sj = (size_t)m->S * m->J;
  if (total_steps) CK(cudaMemcpyAsync(total_steps, m->X.ctotal, sj * 8, cudaMemcpyDeviceToHost, m->st));
  if (throughput) CK(cudaMemcpyAsync(throughput, m->X.cthr, sj * 8, cudaMemcpyDeviceToHost, m->st));
  if (batch_size) CK(cudaMemcpyAsync(batch_size, m->X.cbs, sj * 4, cudaMemcpyDeviceToHost, m->st));
  if (exec_time) CK(cudaMemcpyAsync(exec_time, m->X.last_ex, sj * 8, cudaMemcpyDeviceToHost, m->st));
  if (finish_time) CK(cudaMemcpyAsync(finish_time, m->X.fin, sj * 8, cudaMemcpyDeviceToHost, m->st));
  if (failed_attempts) CK(cudaMemcpyAsync(failed_attempts, m->X.fails, sj, cudaMemcpyDeviceToHost, m->st));
  if (ran) CK(cudaMemcpyAsync(ran, m->X.ranprev, sj, cudaMemcpyDeviceToHost, m->st));
  CK(cudaStreamSynchronize(m->st));
  return 0;
}

}  // extern "C"
