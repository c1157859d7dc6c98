// api.cu — the C-ABI of libswb200.so (see include/swb200.h) and the device-memory bookkeeping.
#include <math.h>
#include <string.h>

#include <string>
#include <vector>

#include "swb_internal.h"

static thread_local std::string g_err;
static int fail(int code, const std::string &msg) { g_err = msg; return code; }

struct swb_ctx {
  int device = 0;
  cudaStream_t st = nullptr;
  // ---- work buffers of a solve
  DBuf prm, res, g, E, c, dbar, rem, ftobj, bfkey, x, bf, nr, w, xmk, bmk;
  DBuf wf_z, wf_x2;
  DBuf sa, su0, sR, sws, scap, sg, snF, snmax, sn, gmask, sncap, seated, scth, sths, sn0, snfc, sRr;
  int want_relaxed = 0;
  int solve_cluster = 8;  // SWB_OPT_SOLVE_CLUSTER
  int aux_async = 0;      // SWB_OPT_ASYNC_AUX: device-output forecast / ensemble calls return without synchronising
  // ---- resident job table (by slot)
  int nslots = 0;
  DBuf t_off, t_E, t_nm, t_g, t_ns, t_ts, t_modes, t_mm, t_amp, s_r0, s_rl, s_cnt, s_vl, s_acc, t_mu, t_sg;
  // Monte-Carlo (GBM) forecast inside swb_round_solve: 0 paths = off (the reference's deterministic forecast)
  int64_t gbm_paths = 0;
  uint64_t gbm_seed = 0;
  int gbm_hmax = 256;
  DBuf ens_z;
  DBuf gv_in, gv_out;     // swb_gavel_round: one staging buffer each way
  DBuf rr_items;          // re-rank local search scratch
  int rr_iters = 400;     // SWB_OPT_RERANK_ITERS (0 = sweep only)
  int rr_restarts = 2;    // SWB_OPT_RERANK_RESTARTS
  DBuf pool_pp, pool_bs;
  int64_t pool_used = 0;
  // holes left by removed jobs in pool_pp / pool_bs: (offset, rows), sorted by offset, adjacent holes merged;
  // swb_job_add takes the first hole that fits, so the pools grow with the LIVE jobs, not with all jobs ever seen
  std::vector<std::pair<int64_t, int64_t>> pool_holes;
  std::vector<int64_t> h_off;
  std::vector<int32_t> h_E;
  // ---- per-call forecast buffers
  DBuf f_remfb, f_bffb, f_ampok, f_ampfb, f_ftest, f_ncal;
  swb::ForecastLaunch last_fc;   // descriptor of the latest forecast (for the calibration commit)
  bool have_fc = false;
  DBuf lp_colp, lp_rowi, lp_val, lp_c, lp_b, lp_Binv, lp_Bm, lp_vec, lp_basis, lp_where, lp_x, lp_out;   // swb_lp_solve
  DBuf ax_p, ax_t, ax_wt, ax_u, ax_v, ax_spc, ax_c4r, ax_r4c, ax_path, ax_sc, ax_sr, ax_out;   // swb_allox_assign
  DBuf pol_coef, pol_sf, pol_t, pol_n, pol_den, pol_x, pol_out;          // swb_policy_pooled
  DBuf het_a, het_N, het_x;                                                 // swb_policy_hetero
  DBuf mc_R0, mc_mu, mc_sigma, mc_H, mc_out;                                 // swb_gbm_forecast
  DBuf m_theta, m_rowp, m_colload, m_colscale, m_price, m_obj, m_X, m_rate, m_E, m_c, m_Gw;
  DBuf m_rowprev, m_mj, m_om, m_colprev, m_pi, m_Xc, m_cc, m_pws;   // PDHG state; m_cc = the coarse level's column arrays
  static constexpr int MEV = 32;           // event pairs around the last MEV/2 dense passes of swb_market_pgd
  cudaEvent_t mev[MEV] = {};
  // CUDA events around the two kernels of the latest solve pass (bench.py's roofline)
  cudaEvent_t ev[3] = {nullptr, nullptr, nullptr};
  int last_passes = 0;
  PinBuf h_res;     // pinned staging for the scalar results
  PinBuf h_stage;   // pinned staging of the per-call inputs / outputs of swb_round_solve / swb_forecast
  DBuf f_in;        // device arena of the per-call forecast inputs (one H2D copy)
};

extern "C" {

void swb_destroy(swb_ctx *c);
int swb_version(void) { return 101; }
const char *swb_last_error(void) { return g_err.c_str(); }
int swb_set_error(int code, const char *msg) { return fail(code, msg ? msg : ""); }

int swb_create(swb_ctx **out, int device) {
  if (!out) return fail(SWB_ERR_ARG, "swb_create: out is null");
  int ndev = 0;
  CK(cudaGetDeviceCount(&ndev));
  if (ndev <= 0) return fail(SWB_ERR_CUDA, "swb_create: no CUDA device (this library has no CPU path)");
  if (device < 0 || device >= ndev) return fail(SWB_ERR_ARG, "swb_create: bad device index");
  CK(cudaSetDevice(device));
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, device));
  if (prop.major < 10)
    return fail(SWB_ERR_CUDA, "swb_create: libswb200 is built for sm_100a only (Blackwell B200)");
  swb_ctx *c = new swb_ctx();
  c->device = device;
  cudaError_t e = cudaStreamCreateWithFlags(&c->st, cudaStreamNonBlocking);
  for (int i = 0; i < 3 && e == cudaSuccess; ++i) e = cudaEventCreate(&c->ev[i]);
  for (int i = 0; i < swb_ctx::MEV && e == cudaSuccess; ++i) e = cudaEventCreate(&c->mev[i]);
  if (e != cudaSuccess) {
    swb_destroy(c);      // releases whatever was created
    return fail(SWB_ERR_CUDA, std::string("swb_create: ") + cudaGetErrorString(e));
  }
  *out = c;
  return 0;
}

void swb_destroy(swb_ctx *c) {
  if (!c) return;
  cudaSetDevice(c->device);
  for (int i = 0; i < 3; ++i) if (c->ev[i]) cudaEventDestroy(c->ev[i]);
  for (int i = 0; i < swb_ctx::MEV; ++i) if (c->mev[i]) cudaEventDestroy(c->mev[i]);
  if (c->st) cudaStreamDestroy(c->st);
  delete c;      // the buffers free themselves
}

void *swb_stream(swb_ctx *c) { return c ? (void *)c->st : nullptr; }
int swb_sync(swb_ctx *c) {
  if (!c) return fail(SWB_ERR_ARG, "null ctx");
  CK(cudaStreamSynchronize(c->st));
  return 0;
}

static int check_params(const swb_params *p, int S, int J) {
  if (J <= 0 || J > SWB_MAX_J) return fail(SWB_ERR_ARG, "J must be in [1, 8192]");
  for (int s = 0; s < S; ++s) {
    if (p[s].future_rounds <= 0 || p[s].future_rounds > SWB_MAX_T)
      return fail(SWB_ERR_ARG, "future_rounds must be in [1, 128]");
    if (p[s].ngpus <= 0) return fail(SWB_ERR_ARG, "ngpus must be positive");
    if (p[s].nbases < 2 || p[s].nbases > 9) return fail(SWB_ERR_ARG, "nbases must be in [2,9]");
    if (!(p[s].round_duration > 0.0)) return fail(SWB_ERR_ARG, "round_duration must be positive");
    if (!(p[s].k > 0.0)) return fail(SWB_ERR_ARG, "k must be positive (shockwave.py:67)");
  }
  return 0;
}

static int ensure_scratch(swb_ctx *c, size_t n) {
  CK(c->sa.need(n * 8, c->st));   CK(c->su0.need(n * 8, c->st)); CK(c->sR.need(n * 8, c->st));
  CK(c->sws.need(n * 8, c->st));  CK(c->scap.need(n * 8, c->st));
  CK(c->sg.need(n, c->st));       CK(c->snF.need(n, c->st));     CK(c->snmax.need(n, c->st));
  CK(c->sn.need(n, c->st));       CK(c->w.need(n * 8, c->st));
  CK(c->sncap.need(n, c->st));    CK(c->seated.need(n * 4, c->st));
  CK(c->snfc.need(n * 8, c->st));
  return 0;
}

// common tail: launch solve + place on device-resident inputs
static int run_solve(swb_ctx *c, int S, int J, int per_scn, const swb_params *h_prm, const int32_t *g,
                     const int32_t *E, const int32_t *cc, const double *dbar, const double *rem,
                     const double *ftobj, const double *bfkey, const double *rem_fb,
                     const double *bfkey_fb, uint8_t *x, uint8_t *bf, int32_t *nr, double *weights,
                     int32_t *ncal = nullptr, unsigned long long *xmask = nullptr,
                     unsigned long long *bfmask = nullptr) {
  const size_t n = (size_t)S * J;
  int rc = ensure_scratch(c, n);
  if (rc) return rc;
  CK(c->res.need(sizeof(swb_result) * S, c->st));
  CK(c->prm.upload(h_prm, sizeof(swb_params) * S, c->st));
  if (J > SWB_SMEM_JOBS) {
    CK(c->gmask.need(n * 4 * sizeof(unsigned long long), c->st));
    CK(c->scth.need(n * 8, c->st)); CK(c->sRr.need(n * 8, c->st)); CK(c->sths.need(n * SWB_MAX_BASES * 4, c->st));
    CK(c->sn0.need(n * SWB_MAX_BASES, c->st));
  }
  swb::SolveLaunch L;
  L.S = S; L.J = J; L.per_scn = per_scn; L.jobs_in_smem = (J <= SWB_SMEM_JOBS) ? 1 : 0;
  L.prm = c->prm.as<swb_params>();
  L.g = g; L.E = E; L.c = cc; L.dbar = dbar; L.rem = rem; L.ftobj = ftobj; L.rem_fb = rem_fb;
  L.sc_a = c->sa.as<double>(); L.sc_u0 = c->su0.as<double>(); L.sc_R = c->sR.as<double>();
  L.sc_ws = c->sws.as<double>(); L.sc_cap = c->scap.as<double>();
  L.sc_g = c->sg.as<uint8_t>(); L.sc_nF = c->snF.as<uint8_t>(); L.sc_nmax = c->snmax.as<uint8_t>();
  L.sc_n = c->sn.as<uint8_t>();
  L.sc_cth = c->scth.as<double>(); L.sc_Rr = c->sRr.as<double>(); L.sc_ths = c->sths.as<float>(); L.sc_n0 = c->sn0.as<uint8_t>();
  L.weights = weights ? weights : c->w.as<double>();
  L.res = c->res.as<swb_result>();
  L.ncap = c->sncap.as<uint8_t>();
  L.sc_nfc = c->snfc.as<double>(); L.want_relaxed = c->want_relaxed;
  L.cluster = c->solve_cluster;
  CK(cudaMemsetAsync(c->sncap.p, 0xff, n, c->st));
  swb::PlaceLaunch P;
  P.S = S; P.J = J; P.per_scn = per_scn; P.prm = L.prm; P.bfkey = bfkey; P.bfkey_fb = bfkey_fb;
  P.sc_a = L.sc_a; P.sc_u0 = L.sc_u0; P.sc_R = L.sc_R; P.sc_ws = L.sc_ws; P.sc_cap = L.sc_cap;
  P.sc_g = L.sc_g; P.sc_n = L.sc_n; P.sc_nmax = L.sc_nmax; P.weights = L.weights; P.E = E; P.c = cc; P.dbar = dbar;
  P.x = x; P.backfill = bf; P.nrounds = nr ? nr : c->seated.as<int32_t>(); P.ncal = ncal; P.res = L.res;
  P.xmask = xmask; P.bfmask = bfmask; P.ncap = c->sncap.as<uint8_t>();
  P.plan = swb::plan_place(S, J, h_prm[0].future_rounds, c->rr_iters, c->solve_cluster);
  if (P.plan.rerank) CK(c->rr_items.need(P.plan.rr_bytes, c->st));
  P.rr_items = c->rr_items.p; P.rr_iters = c->rr_iters; P.rr_restarts = c->rr_restarts;
  CK(c->h_res.need(sizeof(swb_result) * S));
  const swb_result *hres = c->h_res.as<swb_result>();
  for (int pass = 0; pass < SWB_MAX_REPLAN + 1; ++pass) {
    CK(cudaEventRecord(c->ev[0], c->st));
    CK(swb::launch_solve(L, c->st, h_prm[0].nbases));
    CK(cudaEventRecord(c->ev[1], c->st));
    CK(swb::launch_place(P, c->st, c->gmask.as<unsigned long long>()));
    CK(cudaEventRecord(c->ev[2], c->st));
    c->last_passes = pass + 1;
    CK(cudaMemcpyAsync(c->h_res.p, c->res.p, sizeof(swb_result) * S, cudaMemcpyDeviceToHost, c->st));
    CK(cudaStreamSynchronize(c->st));
    int shortf = 0;
    for (int s = 0; s < S; ++s) shortf += hres[s].shortfall;
    if (shortf == 0 || pass == SWB_MAX_REPLAN) break;
    // place_kernel has already written the tighter per-job caps for the next pass (packing feedback)
  }
  return 0;
}

int swb_solve(swb_ctx *c, const swb_solve_args *a) {
  if (!c || !a) return fail(SWB_ERR_ARG, "swb_solve: null argument");
  if (a->S <= 0) return fail(SWB_ERR_ARG, "swb_solve: S must be positive");
  if (!a->prm || !a->res || !a->g || !a->E || !a->c || !a->dbar || !a->rem || !a->ftobj)
    return fail(SWB_ERR_ARG, "swb_solve: missing input pointer");
  int rc = check_params(a->prm, a->S, a->J);
  if (rc) return rc;
  CK(cudaSetDevice(c->device));
  const int S = a->S, J = a->J, T = a->prm[0].future_rounds;
  for (int s = 1; s < S; ++s)
    if (a->prm[s].future_rounds != T || a->prm[s].nbases != a->prm[0].nbases)
      return fail(SWB_ERR_ARG, "swb_solve: all scenarios of one call must share future_rounds and nbases");
  const size_t nj = a->per_scenario_jobs ? (size_t)S * J : (size_t)J;
  const size_t nx = (size_t)S * J * T;
  const int32_t *g, *E, *cc;
  const double *dbar, *rem, *ftobj, *bfkey;
  uint8_t *x, *bf;
  int32_t *nr;
  double *w;
  unsigned long long *xmk = nullptr, *bmk = nullptr;
  if (!a->on_device) {
    // gang widths are kept as bytes on the device (solve.cu, place.cu): reject what does not fit instead of
    // truncating it (on_device inputs are checked by the kernel itself, which reports SWB_ERR_ARG through res)
    for (size_t i = 0; i < nj; ++i)
      if (a->g[i] < 1 || a->g[i] > 255) return fail(SWB_ERR_ARG, "swb_solve: gang width g[j] must be in [1, 255]");
  }
  if (a->on_device) {
    xmk = (unsigned long long *)a->xmask; bmk = (unsigned long long *)a->bfmask;
    g = a->g; E = a->E; cc = a->c; dbar = a->dbar; rem = a->rem; ftobj = a->ftobj;
    bfkey = a->bfkey ? a->bfkey : a->rem;
    x = a->x; bf = a->backfill; nr = a->nrounds; w = a->weights;
  } else {
    CK(c->g.upload(a->g, nj * 4, c->st));
    CK(c->E.upload(a->E, nj * 4, c->st));
    CK(c->c.upload(a->c, nj * 4, c->st));
    CK(c->dbar.upload(a->dbar, nj * 8, c->st));
    CK(c->rem.upload(a->rem, nj * 8, c->st));
    CK(c->ftobj.upload(a->ftobj, nj * 8, c->st));
    CK(c->bfkey.upload(a->bfkey ? a->bfkey : a->rem, nj * 8, c->st));
    g = c->g.as<int32_t>(); E = c->E.as<int32_t>(); cc = c->c.as<int32_t>();
    dbar = c->dbar.as<double>(); rem = c->rem.as<double>(); ftobj = c->ftobj.as<double>();
    bfkey = c->bfkey.as<double>();
    x = nullptr; bf = nullptr; nr = nullptr; w = nullptr;
    if (a->x) { CK(c->x.need(nx, c->st)); x = c->x.as<uint8_t>(); }
    if (a->backfill) { CK(c->bf.need(nx, c->st)); bf = c->bf.as<uint8_t>(); }
    if (a->nrounds) { CK(c->nr.need((size_t)S * J * 4, c->st)); nr = c->nr.as<int32_t>(); }
    if (a->xmask) { CK(c->xmk.need((size_t)S * J * 16, c->st)); xmk = c->xmk.as<unsigned long long>(); }
    if (a->bfmask) { CK(c->bmk.need((size_t)S * J * 16, c->st)); bmk = c->bmk.as<unsigned long long>(); }
  }
  rc = run_solve(c, S, J, a->per_scenario_jobs, a->prm, g, E, cc, dbar, rem, ftobj, bfkey, nullptr,
                 nullptr, x, bf, nr, w, nullptr, xmk, bmk);
  if (rc) return rc;
  CK(cudaMemcpyAsync(c->h_res.p, c->res.p, sizeof(swb_result) * S, cudaMemcpyDeviceToHost, c->st));
  if (!a->on_device) {
    if (a->x) CK(cudaMemcpyAsync(a->x, x, nx, cudaMemcpyDeviceToHost, c->st));
    if (a->backfill) CK(cudaMemcpyAsync(a->backfill, bf, nx, cudaMemcpyDeviceToHost, c->st));
    if (a->nrounds) CK(cudaMemcpyAsync(a->nrounds, nr, (size_t)S * J * 4, cudaMemcpyDeviceToHost, c->st));
    if (a->weights)
      CK(cudaMemcpyAsync(a->weights, c->w.p, (size_t)S * J * 8, cudaMemcpyDeviceToHost, c->st));
    if (a->xmask) CK(cudaMemcpyAsync(a->xmask, xmk, (size_t)S * J * 16, cudaMemcpyDeviceToHost, c->st));
    if (a->bfmask) CK(cudaMemcpyAsync(a->bfmask, bmk, (size_t)S * J * 16, cudaMemcpyDeviceToHost, c->st));
  }
  CK(cudaStreamSynchronize(c->st));
  memcpy(a->res, c->h_res.p, sizeof(swb_result) * S);
  for (int s = 0; s < S; ++s)
    if (a->res[s].flags & 1) return fail(SWB_ERR_ARG, "swb_solve: gang width g[j] must be in [1, 255] (device input)");
  int any_fb = 0;
  for (int s = 0; s < S; ++s) any_fb |= (a->res[s].status == SWB_ST_FALLBACK);
  return any_fb ? SWB_ST_FALLBACK : SWB_ST_OK;
}

// ---- resident job table -------------------------------------------------------------------------
// the per-slot scalars of one job, passed BY VALUE as the kernel parameter: one launch writes the whole row
// (no staging buffer, nothing to keep alive, no stream synchronize on the add path)
struct JobRow {
  int64_t off;
  int32_t slot, E, nmodes, g;
  double nsamples, tsubmit, mu, sigma;
  int32_t modes[SWB_MAX_MODES];
  double modemean[SWB_MAX_MODES];
};
struct JobTablePtrs {
  int64_t *off; int32_t *E, *nm, *g; double *ns, *ts; int32_t *modes; double *mm, *amp; int32_t *cnt; double *acc;
  double *mu, *sg;
};
__global__ void job_row_kernel(JobRow r, JobTablePtrs t) {
  const int i = threadIdx.x;
  if (i < SWB_MAX_MODES) {
    t.modes[(size_t)r.slot * SWB_MAX_MODES + i] = r.modes[i];
    t.mm[(size_t)r.slot * SWB_MAX_MODES + i] = r.modemean[i];
  }
  if (i == 0) {
    t.off[r.slot] = r.off; t.E[r.slot] = r.E; t.nm[r.slot] = r.nmodes; t.g[r.slot] = r.g;
    t.ns[r.slot] = r.nsamples; t.ts[r.slot] = r.tsubmit;
    t.amp[r.slot] = 1.0; t.cnt[r.slot] = 0; t.acc[r.slot] = 0.0;
    t.mu[r.slot] = r.mu; t.sg[r.slot] = r.sigma;
  }
}
__global__ void job_gbm_kernel(int slot, double mu, double sigma, double *tmu, double *tsg) {
  tmu[slot] = mu; tsg[slot] = sigma;
}

static int ensure_slots(swb_ctx *c, int nslots) {
  if (nslots <= c->nslots) return 0;
  size_t n = (size_t)nslots;
  CK(c->t_off.need(n * 8, c->st, true)); CK(c->t_E.need(n * 4, c->st, true));
  CK(c->t_nm.need(n * 4, c->st, true));  CK(c->t_g.need(n * 4, c->st, true));
  CK(c->t_ns.need(n * 8, c->st, true));  CK(c->t_ts.need(n * 8, c->st, true));
  CK(c->t_modes.need(n * 4 * SWB_MAX_MODES, c->st, true));
  CK(c->t_mm.need(n * 8 * SWB_MAX_MODES, c->st, true));
  CK(c->t_amp.need(n * 8, c->st, true));
  CK(c->s_r0.need(n * 4, c->st, true)); CK(c->s_rl.need(n * 4, c->st, true));
  CK(c->s_cnt.need(n * 4, c->st, true)); CK(c->s_vl.need(n * 8, c->st, true));
  CK(c->s_acc.need(n * 8, c->st, true));
  CK(c->t_mu.need(n * 8, c->st, true)); CK(c->t_sg.need(n * 8, c->st, true));
  c->nslots = nslots;
  c->h_off.resize(n, -1);
  c->h_E.resize(n, 0);
  return 0;
}

int swb_job_add(swb_ctx *c, int32_t slot, int32_t nworkers, int32_t epochs, double epoch_nsamples,
                double timestamp_submit, const double *pre, const int32_t *bs) {
  if (!c || !pre || !bs) return fail(SWB_ERR_ARG, "swb_job_add: null argument");
  if (slot < 0 || epochs <= 0) return fail(SWB_ERR_ARG, "swb_job_add: bad slot / epochs");
  if (nworkers <= 0 || nworkers > 255) return fail(SWB_ERR_ARG, "swb_job_add: nworkers must be in [1,255]");
  CK(cudaSetDevice(c->device));
  int rc = ensure_slots(c, slot + 1);
  if (rc) return rc;
  if (c->h_off[slot] >= 0)
    return fail(SWB_ERR_STATE, "swb_job_add: slot is occupied (swb_job_remove it first)");
  // host-side digest of the static profile: prefix sums (sequential, like the reference's running
  // `preprofiled_time_range += duration`, JobMetaData.py:253-257), sorted bs modes
  // (JobMetaData.py:296), per-mode mean duration (JobMetaData.py:304-312, pairwise like np.mean).
  std::vector<double> pp((size_t)epochs + 1);
  pp[0] = 0.0;
  for (int e = 0; e < epochs; ++e) pp[e + 1] = pp[e] + pre[e];
  std::vector<int32_t> modes;
  for (int e = 0; e < epochs; ++e) {
    bool seen = false;
    for (int32_t m : modes) if (m == bs[e]) { seen = true; break; }
    if (!seen) modes.push_back(bs[e]);
  }
  if ((int)modes.size() > SWB_MAX_MODES) return fail(SWB_ERR_ARG, "swb_job_add: more than 16 batch-size modes");
  for (size_t i = 1; i < modes.size(); ++i)
    for (size_t k = i; k > 0 && modes[k - 1] > modes[k]; --k) std::swap(modes[k - 1], modes[k]);
  int32_t hm[SWB_MAX_MODES] = {0};
  double hmm[SWB_MAX_MODES] = {0};
  std::vector<double> tmp;
  for (size_t m = 0; m < modes.size(); ++m) {
    hm[m] = modes[m];
    tmp.clear();
    for (int e = 0; e < epochs; ++e) if (bs[e] == modes[m]) tmp.push_back(pre[e]);
    // numpy's pairwise summation (blocks of 8 accumulators below 128 elements)
    struct PW {
      static double sum(const double *a, size_t n) {
        if (n < 8) { double r = 0.0; for (size_t i = 0; i < n; ++i) r += a[i]; return r; }
        if (n <= 128) {
          double r[8];
          for (int i = 0; i < 8; ++i) r[i] = a[i];
          size_t i = 8;
          for (; i + 8 <= n; i += 8) for (int k = 0; k < 8; ++k) r[k] += a[i + k];
          double res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
          for (; i < n; ++i) res += a[i];
          return res;
        }
        size_t n2 = n / 2;
        n2 -= n2 % 8;
        return sum(a, n2) + sum(a + n2, n - n2);
      }
    };
    hmm[m] = PW::sum(tmp.data(), tmp.size()) / (double)tmp.size();
  }
  const size_t rows = (size_t)epochs + 1;
  // first hole that fits (left by removed jobs), else the end of the pool
  int64_t off = -1;
  for (size_t h = 0; h < c->pool_holes.size(); ++h) {
    if (c->pool_holes[h].second >= (int64_t)rows) {
      off = c->pool_holes[h].first;
      c->pool_holes[h].first += (int64_t)rows;
      c->pool_holes[h].second -= (int64_t)rows;
      if (c->pool_holes[h].second == 0) c->pool_holes.erase(c->pool_holes.begin() + h);
      break;
    }
  }
  if (off < 0) {
    off = c->pool_used;
    CK(c->pool_pp.need((off + rows) * 8, c->st, true));
    CK(c->pool_bs.need((off + rows) * 4, c->st, true));
    c->pool_used += rows;
  }
  // pageable sources: cudaMemcpyAsync returns once they are staged, so the vectors may die with this frame
  CK(cudaMemcpyAsync(c->pool_pp.as<double>() + off, pp.data(), rows * 8, cudaMemcpyHostToDevice, c->st));
  CK(cudaMemcpyAsync(c->pool_bs.as<int32_t>() + off, bs, (size_t)epochs * 4, cudaMemcpyHostToDevice, c->st));
  c->h_off[slot] = off;
  c->h_E[slot] = epochs;
  JobRow r;
  r.off = off; r.slot = slot; r.E = epochs; r.nmodes = (int32_t)modes.size(); r.g = nworkers;
  r.nsamples = epoch_nsamples; r.tsubmit = timestamp_submit;
  // default volatility model of the job (only read when the GBM forecast is switched on): no drift, sigma = the
  // relative spread of the pre-profiled epoch durations INSIDE their batch-size modes — zero for the profiles the
  // reference generates (utils.py:1350-1430: one duration per mode), so the default reproduces the reference
  {
    double ss = 0.0, tot = 0.0;
    for (int e = 0; e < epochs; ++e) {
      size_t m = 0;
      while (m + 1 < modes.size() && modes[m] != bs[e]) ++m;
      const double d = pre[e] - hmm[m];
      ss += d * d; tot += pre[e];
    }
    const double mean = tot / (double)epochs;
    r.mu = 0.0;
    r.sigma = mean > 0.0 ? sqrt(ss / (double)epochs) / mean : 0.0;
    if (r.sigma < 1e-12) r.sigma = 0.0;
  }
  memcpy(r.modes, hm, sizeof(hm)); memcpy(r.modemean, hmm, sizeof(hmm));
  JobTablePtrs t;
  t.off = c->t_off.as<int64_t>(); t.E = c->t_E.as<int32_t>(); t.nm = c->t_nm.as<int32_t>(); t.g = c->t_g.as<int32_t>();
  t.ns = c->t_ns.as<double>(); t.ts = c->t_ts.as<double>(); t.modes = c->t_modes.as<int32_t>();
  t.mm = c->t_mm.as<double>(); t.amp = c->t_amp.as<double>(); t.cnt = c->s_cnt.as<int32_t>(); t.acc = c->s_acc.as<double>();
  t.mu = c->t_mu.as<double>(); t.sg = c->t_sg.as<double>();
  job_row_kernel<<<1, 32, 0, c->st>>>(r, t);
  CK(cudaGetLastError());
  c->have_fc = false;      // the tables may have moved: a pending forecast can no longer be committed
  return 0;
}

int swb_job_remove(swb_ctx *c, int32_t slot) {
  if (!c || slot < 0 || slot >= c->nslots || c->h_off[slot] < 0)
    return fail(SWB_ERR_ARG, "swb_job_remove: unknown slot");
  // return the job's rows to the hole list (sorted by offset, neighbours merged); a hole that reaches the end
  // of the pool shrinks pool_used instead
  const int64_t off = c->h_off[slot], rows = (int64_t)c->h_E[slot] + 1;
  auto &H = c->pool_holes;
  size_t pos = 0;
  while (pos < H.size() && H[pos].first < off) ++pos;
  H.insert(H.begin() + pos, std::make_pair(off, rows));
  if (pos + 1 < H.size() && H[pos].first + H[pos].second == H[pos + 1].first) {
    H[pos].second += H[pos + 1].second; H.erase(H.begin() + pos + 1);
  }
  if (pos > 0 && H[pos - 1].first + H[pos - 1].second == H[pos].first) {
    H[pos - 1].second += H[pos].second; H.erase(H.begin() + pos);
  }
  if (!H.empty() && H.back().first + H.back().second == c->pool_used) { c->pool_used = H.back().first; H.pop_back(); }
  c->h_off[slot] = -1;
  c->have_fc = false;
  return 0;
}

int swb_job_set_gbm(swb_ctx *c, int32_t slot, double mu, double sigma) {
  if (!c || slot < 0 || slot >= c->nslots || c->h_off[slot] < 0)
    return fail(SWB_ERR_ARG, "swb_job_set_gbm: unknown slot");
  if (!(sigma >= 0.0) || !isfinite(mu) || !isfinite(sigma))
    return fail(SWB_ERR_ARG, "swb_job_set_gbm: need finite mu and sigma >= 0");
  CK(cudaSetDevice(c->device));
  job_gbm_kernel<<<1, 1, 0, c->st>>>(slot, mu, sigma, c->t_mu.as<double>(), c->t_sg.as<double>());
  CK(cudaGetLastError());
  return 0;
}

int swb_job_table_stats(swb_ctx *c, int64_t *used_rows, int64_t *hole_rows) {
  if (!c) return fail(SWB_ERR_ARG, "null ctx");
  int64_t h = 0;
  for (auto &p : c->pool_holes) h += p.second;
  if (used_rows) *used_rows = c->pool_used;
  if (hole_rows) *hole_rows = h;
  return 0;
}

static int run_forecast(swb_ctx *c, const swb_params *prm, const swb_round_args *a) {
  const int J = a->J;
  for (int j = 0; j < J; ++j) {
    const int s = a->slots[j];
    if (s < 0 || s >= c->nslots || c->h_off[s] < 0) return fail(SWB_ERR_ARG, "unknown job slot");
    if (a->epoch_progress[j] < 0 || a->epoch_progress[j] > c->h_E[s])
      return fail(SWB_ERR_ARG, "epoch_progress out of range (JobMetaData.py:164)");
  }
  CK(c->g.need(J * 4, c->st)); CK(c->E.need(J * 4, c->st)); CK(c->c.need(J * 4, c->st));
  CK(c->dbar.need(J * 8, c->st)); CK(c->rem.need(J * 8, c->st)); CK(c->ftobj.need(J * 8, c->st));
  CK(c->bfkey.need(J * 8, c->st)); CK(c->f_remfb.need(J * 8, c->st)); CK(c->f_bffb.need(J * 8, c->st));
  CK(c->f_ampok.need(J * 8, c->st)); CK(c->f_ampfb.need(J * 8, c->st)); CK(c->f_ftest.need(J * 8, c->st));
  // the four per-call input arrays (20 bytes per job) travel as ONE copy from pinned staging: a cudaMemcpyAsync from
  // pageable memory is a staged, synchronous copy of its own (every API call ends with a stream sync, so the staging
  // buffer is free again when the next call starts)
  const size_t Jz = (size_t)J;
  CK(c->h_stage.need(84 * Jz + 64));
  unsigned char *hs = c->h_stage.as<unsigned char>();
  memcpy(hs, a->meas_nsamples, 8 * Jz);
  memcpy(hs + 8 * Jz, a->slots, 4 * Jz);
  memcpy(hs + 12 * Jz, a->epoch_progress, 4 * Jz);
  memcpy(hs + 16 * Jz, a->meas_end_round, 4 * Jz);
  CK(c->f_in.upload(hs, 20 * Jz, c->st));
  unsigned char *din = reinterpret_cast<unsigned char *>(c->f_in.p);
  swb::ForecastLaunch F;
  F.J = J; F.reestimate_share = a->reestimate_share; F.round_ptr = prm->round_ptr; F.ngpus = prm->ngpus;
  F.gavel_round_duration = a->gavel_round_duration;
  F.meas_ns = reinterpret_cast<double *>(din); F.slots = reinterpret_cast<int32_t *>(din + 8 * Jz);
  F.progress = reinterpret_cast<int32_t *>(din + 12 * Jz); F.meas_end = reinterpret_cast<int32_t *>(din + 16 * Jz);
  F.tab_off = c->t_off.as<int64_t>(); F.tab_E = c->t_E.as<int32_t>(); F.tab_nmodes = c->t_nm.as<int32_t>();
  F.tab_g = c->t_g.as<int32_t>(); F.tab_nsamples = c->t_ns.as<double>(); F.tab_tsubmit = c->t_ts.as<double>();
  F.tab_modes = c->t_modes.as<int32_t>(); F.tab_modemean = c->t_mm.as<double>(); F.tab_amp = c->t_amp.as<double>();
  F.ss_r0 = c->s_r0.as<int32_t>(); F.ss_rlast = c->s_rl.as<int32_t>(); F.ss_cnt = c->s_cnt.as<int32_t>();
  F.ss_vlast = c->s_vl.as<double>(); F.ss_acc = c->s_acc.as<double>();
  F.pool_prefix = c->pool_pp.as<double>(); F.pool_bs = c->pool_bs.as<int32_t>();
  F.dbar = c->dbar.as<double>(); F.rem = c->rem.as<double>(); F.ftobj = c->ftobj.as<double>();
  F.bfkey = c->bfkey.as<double>(); F.ftest = c->f_ftest.as<double>();
  F.rem_fb = c->f_remfb.as<double>(); F.bfkey_fb = c->f_bffb.as<double>();
  F.amp_ok = c->f_ampok.as<double>(); F.amp_fb = c->f_ampfb.as<double>();
  F.g_out = c->g.as<int32_t>(); F.E_out = c->E.as<int32_t>(); F.c_out = c->c.as<int32_t>();
  CK(swb::launch_forecast(F, c->st));
  c->last_fc = F;
  c->have_fc = true;
  return 0;
}

int swb_round_solve(swb_ctx *c, const swb_params *prm, const swb_round_args *a) {
  if (!c || !prm || !a || !a->slots || !a->epoch_progress || !a->meas_nsamples || !a->meas_end_round ||
      !a->res)
    return fail(SWB_ERR_ARG, "swb_round_solve: null argument");
  int rc = check_params(prm, 1, a->J);
  if (rc) return rc;
  CK(cudaSetDevice(c->device));
  const int J = a->J, T = prm->future_rounds;
  rc = run_forecast(c, prm, a);
  if (rc) return rc;
  if (c->gbm_paths > 0) {
    // Monte-Carlo forecast on the device, between the deterministic forecast and the solve (no host round trip):
    // R0 = the Dirichlet forecast just computed, horizon min(E - c, Hmax) epochs, per-job (mu, sigma) from the table
    CK(c->mc_out.need((size_t)J * 16, c->st));
    swb::GbmLaunch Gm;
    Gm.J = J; Gm.P_local = c->gbm_paths; Gm.path_offset = 0; Gm.seed = c->gbm_seed ^ (uint64_t)prm->round_ptr * 0x9E3779B97F4A7C15ull;
    Gm.R0 = c->rem.as<double>(); Gm.mu = nullptr; Gm.sigma = nullptr; Gm.H = nullptr;
    Gm.out = c->mc_out.as<double>();
    Gm.slots = c->last_fc.slots; Gm.Eo = c->E.as<int32_t>(); Gm.co = c->c.as<int32_t>();
    Gm.tab_mu = c->t_mu.as<double>(); Gm.tab_sigma = c->t_sg.as<double>(); Gm.Hmax = c->gbm_hmax;
    CK(swb::launch_gbm(Gm, c->st));
    swb::GbmApplyLaunch Ga;
    Ga.J = J; Ga.P_total = (double)c->gbm_paths; Ga.sums = Gm.out; Ga.slots = Gm.slots;
    Ga.tab_mu = Gm.tab_mu; Ga.tab_sigma = Gm.tab_sigma;
    Ga.rem = c->rem.as<double>(); Ga.rem_fb = c->f_remfb.as<double>();
    Ga.bfkey = c->bfkey.as<double>(); Ga.bfkey_fb = c->f_bffb.as<double>(); Ga.var_out = nullptr;
    CK(swb::launch_gbm_apply(Ga, c->st));
  }
  const size_t nx = (size_t)J * T;
  uint8_t *dx = nullptr, *dbf = nullptr;
  unsigned long long *dxm = nullptr, *dbm = nullptr;
  if (a->x) { CK(c->x.need(nx, c->st)); dx = c->x.as<uint8_t>(); }
  if (a->backfill) { CK(c->bf.need(nx, c->st)); dbf = c->bf.as<uint8_t>(); }
  if (a->xmask) { CK(c->xmk.need((size_t)J * 16, c->st)); dxm = c->xmk.as<unsigned long long>(); }
  if (a->bfmask) { CK(c->bmk.need((size_t)J * 16, c->st)); dbm = c->bmk.as<unsigned long long>(); }
  CK(c->nr.need((size_t)J * 4, c->st));
  CK(c->f_ncal.need((size_t)J * 4, c->st));
  rc = run_solve(c, 1, J, 0, prm, c->g.as<int32_t>(), c->E.as<int32_t>(), c->c.as<int32_t>(),
                 c->dbar.as<double>(), c->rem.as<double>(), c->ftobj.as<double>(), c->bfkey.as<double>(),
                 c->f_remfb.as<double>(), c->f_bffb.as<double>(), dx, dbf,
                 c->nr.as<int32_t>(), nullptr, c->f_ncal.as<int32_t>(), dxm, dbm);
  if (rc) return rc;
  CK(swb::launch_commit_calibration(c->last_fc, c->res.as<swb_result>(), 0, c->f_ncal.as<int32_t>(), c->st));
  CK(cudaMemcpyAsync(c->h_res.p, c->res.p, sizeof(swb_result), cudaMemcpyDeviceToHost, c->st));
  if (a->x) CK(cudaMemcpyAsync(a->x, c->x.p, nx, cudaMemcpyDeviceToHost, c->st));
  if (a->backfill) CK(cudaMemcpyAsync(a->backfill, c->bf.p, nx, cudaMemcpyDeviceToHost, c->st));
  // the packed outputs (84 bytes per job) come back through the pinned staging buffer — truly asynchronous copies and
  // one sync — and are handed to the caller's (pageable) arrays by memcpy
  unsigned char *hs = c->h_stage.as<unsigned char>();
  const size_t Jz = (size_t)J;
  if (a->xmask) CK(cudaMemcpyAsync(hs, dxm, 16 * Jz, cudaMemcpyDeviceToHost, c->st));
  if (a->bfmask) CK(cudaMemcpyAsync(hs + 16 * Jz, dbm, 16 * Jz, cudaMemcpyDeviceToHost, c->st));
  if (a->nrounds) CK(cudaMemcpyAsync(hs + 32 * Jz, c->nr.p, 4 * Jz, cudaMemcpyDeviceToHost, c->st));
  if (a->forecast_out) {   // [6][J] planes: dbar, rem, ftobj, bfkey, rem_fb, bfkey_fb
    unsigned char *fo = hs + 36 * Jz;
    CK(cudaMemcpyAsync(fo, c->dbar.p, 8 * Jz, cudaMemcpyDeviceToHost, c->st));
    CK(cudaMemcpyAsync(fo + 8 * Jz, c->rem.p, 8 * Jz, cudaMemcpyDeviceToHost, c->st));
    CK(cudaMemcpyAsync(fo + 16 * Jz, c->ftobj.p, 8 * Jz, cudaMemcpyDeviceToHost, c->st));
    CK(cudaMemcpyAsync(fo + 24 * Jz, c->bfkey.p, 8 * Jz, cudaMemcpyDeviceToHost, c->st));
    CK(cudaMemcpyAsync(fo + 32 * Jz, c->f_remfb.p, 8 * Jz, cudaMemcpyDeviceToHost, c->st));
    CK(cudaMemcpyAsync(fo + 40 * Jz, c->f_bffb.p, 8 * Jz, cudaMemcpyDeviceToHost, c->st));
  }
  CK(cudaStreamSynchronize(c->st));
  if (a->xmask) memcpy(a->xmask, hs, 16 * Jz);
  if (a->bfmask) memcpy(a->bfmask, hs + 16 * Jz, 16 * Jz);
  if (a->nrounds) memcpy(a->nrounds, hs + 32 * Jz, 4 * Jz);
  if (a->forecast_out) memcpy(a->forecast_out, hs + 36 * Jz, 48 * Jz);
  *a->res = *c->h_res.as<swb_result>();
  return a->res->status == SWB_ST_FALLBACK ? SWB_ST_FALLBACK : SWB_ST_OK;
}

int swb_forecast(swb_ctx *c, const swb_params *prm, const swb_round_args *a, double *dbar, double *rem,
                 double *ftobj, double *bfkey, double *ft_estimate) {
  if (!c || !prm || !a || !a->slots || !a->epoch_progress || !a->meas_nsamples || !a->meas_end_round)
    return fail(SWB_ERR_ARG, "swb_forecast: null argument");
  if (a->J <= 0) return fail(SWB_ERR_ARG, "swb_forecast: J must be positive");
  CK(cudaSetDevice(c->device));
  int rc = run_forecast(c, prm, a);
  if (rc) return rc;
  const int J = a->J;
  if (dbar) CK(cudaMemcpyAsync(dbar, c->dbar.p, J * 8, cudaMemcpyDeviceToHost, c->st));
  if (rem) CK(cudaMemcpyAsync(rem, c->rem.p, J * 8, cudaMemcpyDeviceToHost, c->st));
  if (ftobj) CK(cudaMemcpyAsync(ftobj, c->ftobj.p, J * 8, cudaMemcpyDeviceToHost, c->st));
  if (bfkey) CK(cudaMemcpyAsync(bfkey, c->bfkey.p, J * 8, cudaMemcpyDeviceToHost, c->st));
  if (ft_estimate) CK(cudaMemcpyAsync(ft_estimate, c->f_ftest.p, J * 8, cudaMemcpyDeviceToHost, c->st));
  CK(cudaStreamSynchronize(c->st));
  return 0;
}

int swb_policy_pooled(swb_ctx *c, int32_t mode, int32_t J, double N, const double *coef, const double *sf,
                      const double *t, const double *n, const double *den, double *x, double *objective) {
  if (!c || !coef || !sf || !x) return fail(SWB_ERR_ARG, "swb_policy_pooled: null argument");
  if (J <= 0 || J > SWB_MAX_J) return fail(SWB_ERR_ARG, "swb_policy_pooled: J must be in [1, 8192]");
  if (mode < SWB_POL_MAXMIN || mode > SWB_POL_ISOLATED) return fail(SWB_ERR_ARG, "swb_policy_pooled: bad mode");
  if (mode == SWB_POL_FTF && (!t || !n || !den)) return fail(SWB_ERR_ARG, "swb_policy_pooled: FTF needs t, n, den");
  if (mode == SWB_POL_MTD && !n) return fail(SWB_ERR_ARG, "swb_policy_pooled: MTD needs n");
  CK(cudaSetDevice(c->device));
  const size_t b = (size_t)J * 8;
  CK(c->pol_t.need(b, c->st)); CK(c->pol_n.need(b, c->st)); CK(c->pol_den.need(b, c->st));
  CK(c->pol_x.need(b, c->st)); CK(c->pol_out.need(16, c->st));
  CK(c->pol_coef.upload(coef, b, c->st));
  CK(c->pol_sf.upload(sf, b, c->st));
  if (t) CK(cudaMemcpyAsync(c->pol_t.p, t, b, cudaMemcpyHostToDevice, c->st));
  if (n) CK(cudaMemcpyAsync(c->pol_n.p, n, b, cudaMemcpyHostToDevice, c->st));
  if (den) CK(cudaMemcpyAsync(c->pol_den.p, den, b, cudaMemcpyHostToDevice, c->st));
  swb::PolicyLaunch L;
  L.mode = mode; L.J = J; L.N = N;
  L.coef = c->pol_coef.as<double>(); L.sf = c->pol_sf.as<double>();
  L.t = t ? c->pol_t.as<double>() : nullptr;        // MAXSUM: optional SLO floors
  L.n = n ? c->pol_n.as<double>() : nullptr; L.den = den ? c->pol_den.as<double>() : nullptr;
  L.x = c->pol_x.as<double>(); L.out = c->pol_out.as<double>();
  CK(swb::launch_policy(L, c->st));
  double out[2] = {0.0, 0.0};
  CK(cudaMemcpyAsync(x, c->pol_x.p, b, cudaMemcpyDeviceToHost, c->st));
  CK(cudaMemcpyAsync(out, c->pol_out.p, 16, cudaMemcpyDeviceToHost, c->st));
  CK(cudaStreamSynchronize(c->st));
  if (objective) *objective = out[0];
  return out[1] != 0.0 ? 1 : 0;
}

int swb_policy_hetero(swb_ctx *c, int32_t mode, int32_t J, int32_t W, const double *N, const double *a,
                      const double *sf, const double *t, const double *n, const double *den, double *x,
                      double *objective, int32_t *stats) {
  if (!c || !N || !a || !sf || !x) return fail(SWB_ERR_ARG, "swb_policy_hetero: null argument");
  if (J <= 0 || J > SWB_MAX_J) return fail(SWB_ERR_ARG, "swb_policy_hetero: J must be in [1, 8192]");
  if (W <= 0 || W > 4 || (mode == SWB_POL_MAXSUM && W > 3))
    return fail(SWB_ERR_ARG, "swb_policy_hetero: W must be in [1, 4] (max-sum: [1, 3])");
  if (mode < SWB_POL_MAXMIN || mode > SWB_POL_MAXSUM) return fail(SWB_ERR_ARG, "swb_policy_hetero: bad mode");
  if (mode == SWB_POL_FTF && (!t || !n || !den)) return fail(SWB_ERR_ARG, "swb_policy_hetero: FTF needs t, n, den");
  if (mode == SWB_POL_MTD && !n) return fail(SWB_ERR_ARG, "swb_policy_hetero: MTD needs n");
  for (int w = 0; w < W; ++w)
    if (!(N[w] > 0.0)) return fail(SWB_ERR_ARG, "swb_policy_hetero: every worker type needs capacity > 0 (drop empty types)");
  CK(cudaSetDevice(c->device));
  const size_t b = (size_t)J * 8, bw = b * (size_t)W;
  CK(c->het_x.need(bw, c->st)); CK(c->het_N.need(32, c->st));
  CK(c->pol_t.need(b, c->st)); CK(c->pol_n.need(b, c->st)); CK(c->pol_den.need(b, c->st));
  CK(c->pol_out.need(128, c->st));
  CK(c->het_a.upload(a, bw, c->st));
  CK(cudaMemcpyAsync(c->het_N.p, N, (size_t)W * 8, cudaMemcpyHostToDevice, c->st));
  CK(c->pol_sf.upload(sf, b, c->st));
  if (t) CK(cudaMemcpyAsync(c->pol_t.p, t, b, cudaMemcpyHostToDevice, c->st));
  if (n) CK(cudaMemcpyAsync(c->pol_n.p, n, b, cudaMemcpyHostToDevice, c->st));
  // MAXSUM with SLO floors: t = needed throughput per job, den = instance cost per worker type (W entries)
  if (den) CK(cudaMemcpyAsync(c->pol_den.p, den, mode == SWB_POL_MAXSUM ? (size_t)W * 8 : b, cudaMemcpyHostToDevice, c->st));
  swb::HeteroLaunch L;
  L.mode = mode; L.J = J; L.W = W;
  L.N = c->het_N.as<double>(); L.a = c->het_a.as<double>(); L.sf = c->pol_sf.as<double>();
  L.t = t ? c->pol_t.as<double>() : nullptr; L.n = n ? c->pol_n.as<double>() : nullptr;
  L.den = den ? c->pol_den.as<double>() : nullptr;
  L.x = c->het_x.as<double>(); L.out = c->pol_out.as<double>();
  if (mode == SWB_POL_MAXSUM && ((t != nullptr) != (den != nullptr)))
    return fail(SWB_ERR_ARG, "swb_policy_hetero: MAXSUM SLO floors need both t (needed throughput) and den (cost per type)");
  CK(swb::launch_hetero(L, c->st));
  double out[16] = {0.0};
  CK(cudaMemcpyAsync(x, c->het_x.p, bw, cudaMemcpyDeviceToHost, c->st));
  CK(cudaMemcpyAsync(out, c->pol_out.p, 128, cudaMemcpyDeviceToHost, c->st));
  CK(cudaStreamSynchronize(c->st));
  if (objective) *objective = out[0];
  if (stats) { stats[0] = (int32_t)out[2]; stats[1] = (int32_t)out[3]; }
  return out[1] != 0.0 ? 1 : 0;
}

int swb_policy_waterfill_step(swb_ctx *c, int32_t J, int32_t W, const double *N, const double *thr, const double *sf,
                              const double *prop, const double *lower, const double *mult, double M, double slack,
                              double *x, double *cobj, double *z, int32_t *stats) {
  if (!c || !N || !thr || !sf || !prop || !lower || !mult || !x || !cobj || !z)
    return fail(SWB_ERR_ARG, "swb_policy_waterfill_step: null argument");
  if (J <= 0 || J > SWB_MAX_J) return fail(SWB_ERR_ARG, "swb_policy_waterfill_step: J must be in [1, 8192]");
  if (W <= 0 || W > 3) return fail(SWB_ERR_ARG, "swb_policy_waterfill_step: W must be in [1, 3]");
  if (!(slack >= 1.0)) return fail(SWB_ERR_ARG, "swb_policy_waterfill_step: slack must be >= 1");
  for (int w = 0; w < W; ++w)
    if (!(N[w] > 0.0)) return fail(SWB_ERR_ARG, "swb_policy_waterfill_step: every worker type needs capacity > 0 (drop empty types)");
  for (int j = 0; j < J; ++j)
    if (!(prop[j] > 0.0) || !(mult[j] >= 0.0) || !(sf[j] > 0.0))
      return fail(SWB_ERR_ARG, "swb_policy_waterfill_step: prop and sf must be positive, mult non-negative");
  CK(cudaSetDevice(c->device));
  const size_t b = (size_t)J * 8, bw = b * (size_t)W;
  CK(c->het_x.need(bw, c->st)); CK(c->het_N.need(32, c->st));
  CK(c->pol_out.need(256, c->st)); CK(c->wf_z.need(b, c->st)); CK(c->wf_x2.need(bw, c->st));
  CK(c->het_a.upload(thr, bw, c->st));
  CK(cudaMemcpyAsync(c->het_N.p, N, (size_t)W * 8, cudaMemcpyHostToDevice, c->st));
  CK(c->pol_sf.upload(sf, b, c->st));
  CK(c->pol_t.upload(lower, b, c->st));
  CK(c->pol_n.upload(mult, b, c->st));
  CK(c->pol_den.upload(prop, b, c->st));
  swb::HeteroLaunch L;
  L.mode = SWB_POL_WFILL; L.J = J; L.W = W;
  L.N = c->het_N.as<double>(); L.a = c->het_a.as<double>(); L.sf = c->pol_sf.as<double>();
  L.t = c->pol_t.as<double>(); L.n = c->pol_n.as<double>(); L.den = c->pol_den.as<double>();
  L.x = c->het_x.as<double>(); L.out = c->pol_out.as<double>();
  L.wf_M = M; L.wf_slack = slack;
  CK(swb::launch_hetero(L, c->st));
  // second program on the same stream: the LP's objective stays on the device (out[0]) and moves the lower bounds
  swb::HeteroLaunch Z = L;
  Z.mode = SWB_POL_WFZ; Z.wf_c = c->pol_out.as<double>(); Z.out = c->pol_out.as<double>() + 16;
  Z.x = c->wf_x2.as<double>(); Z.zout = c->wf_z.as<double>();
  CK(swb::launch_hetero(Z, c->st));
  double out[32] = {0.0};
  CK(cudaMemcpyAsync(out, c->pol_out.p, 256, cudaMemcpyDeviceToHost, c->st));
  CK(cudaStreamSynchronize(c->st));
  if (stats) { stats[0] = (int32_t)out[2]; stats[1] = (int32_t)out[3]; stats[2] = (int32_t)out[18]; stats[3] = (int32_t)out[19]; }
  if (out[1] != 0.0) return 1;
  CK(cudaMemcpyAsync(x, c->het_x.p, bw, cudaMemcpyDeviceToHost, c->st));
  CK(cudaMemcpyAsync(z, c->wf_z.p, b, cudaMemcpyDeviceToHost, c->st));
  CK(cudaStreamSynchronize(c->st));
  *cobj = out[0];
  if (out[17] != 0.0) for (int j = 0; j < J; ++j) z[j] = 0.0;     // the bottleneck program found no point: nobody moves
  return 0;
}

int swb_gbm_forecast(swb_ctx *c, int32_t J, const double *R0, const int32_t *H, const double *mu,
                     const double *sigma, int64_t P_local, int64_t path_offset, uint64_t seed, double *out,
                     int32_t out_on_device) {
  if (!c || !R0 || !H || !mu || !sigma || !out) return fail(SWB_ERR_ARG, "swb_gbm_forecast: null argument");
  if (J <= 0 || P_local < 0) return fail(SWB_ERR_ARG, "swb_gbm_forecast: bad J / P_local");
  CK(cudaSetDevice(c->device));
  const size_t b = (size_t)J * 8;
  const int in_dev = (out_on_device & 2) ? 1 : 0;      // bit 1: R0, H, mu, sigma are device pointers as well
  out_on_device &= 1;
  swb::GbmLaunch L;
  L.J = J; L.P_local = P_local; L.path_offset = path_offset; L.seed = seed;
  CK(c->mc_out.need(2 * b, c->st));
  if (in_dev) {
    L.R0 = R0; L.mu = mu; L.sigma = sigma; L.H = H;
  } else {
    CK(c->mc_R0.upload(R0, b, c->st));
    CK(c->mc_mu.upload(mu, b, c->st));
    CK(c->mc_sigma.upload(sigma, b, c->st));
    CK(c->mc_H.upload(H, (size_t)J * 4, c->st));
    L.R0 = c->mc_R0.as<double>(); L.mu = c->mc_mu.as<double>(); L.sigma = c->mc_sigma.as<double>();
    L.H = c->mc_H.as<int32_t>();
  }
  L.slots = nullptr; L.Eo = nullptr; L.co = nullptr; L.tab_mu = nullptr; L.tab_sigma = nullptr; L.Hmax = 0;
  L.out = out_on_device ? out : c->mc_out.as<double>();
  CK(cudaEventRecord(c->ev[0], c->st));
  CK(swb::launch_gbm(L, c->st));
  CK(cudaEventRecord(c->ev[1], c->st));
  CK(cudaEventRecord(c->ev[2], c->st));
  if (!out_on_device) CK(cudaMemcpyAsync(out, c->mc_out.p, 2 * b, cudaMemcpyDeviceToHost, c->st));
  if (!(c->aux_async && out_on_device && in_dev)) CK(cudaStreamSynchronize(c->st));
  return 0;
}

int swb_gavel_round(swb_ctx *c, const swb_gavel_round_args *a) {
  if (!c || !a) return fail(SWB_ERR_ARG, "swb_gavel_round: null argument");
  const int J = a->J, W = a->W;
  if (J <= 0 || J > SWB_MAX_J || W <= 0 || W > 8) return fail(SWB_ERR_ARG, "swb_gavel_round: need J in [1,8192], W in [1,8]");
  if (!a->type_order || !a->capacity || !a->alloc || !a->job_time || !a->thr || !a->deficit || !a->worker_time ||
      !a->sf || !a->nworkers || !a->worker_ids || !a->prev_type || !a->prev_off || !a->prev_local || !a->prio ||
      !a->n_sel || !a->sel_jobs || !a->n_assigned || !a->assign_job || !a->assign_off || !a->assign_workers)
    return fail(SWB_ERR_ARG, "swb_gavel_round: missing pointer");
  int totw = 0, maxw = 0;
  for (int t = 0; t < W; ++t) {
    if (a->nworkers[t] < 0 || a->nworkers[t] > 8192) return fail(SWB_ERR_ARG, "swb_gavel_round: <= 8192 workers per type");
    totw += a->nworkers[t]; if (a->nworkers[t] > maxw) maxw = a->nworkers[t];
    if (a->type_order[t] < 0 || a->type_order[t] >= W) return fail(SWB_ERR_ARG, "swb_gavel_round: bad type_order");
  }
  const int nprev = a->prev_off[J];
  for (int j = 0; j < J; ++j) {
    if (a->sf[j] <= 0) return fail(SWB_ERR_ARG, "swb_gavel_round: scale factors must be positive");
    if (a->prev_off[j + 1] < a->prev_off[j]) return fail(SWB_ERR_ARG, "swb_gavel_round: prev_off must be non-decreasing");
  }
  CK(cudaSetDevice(c->device));
  // one staging buffer each way: [doubles | int32s | bytes]
  const size_t JW = (size_t)J * W;
  const size_t nd_in = 4 * JW + W;                                  // alloc, job_time, thr, deficit, worker_time
  const size_t ni_in = 2 * (size_t)W + J + W + totw + J + (J + 1) + (size_t)nprev;
  const size_t in_bytes = nd_in * 8 + ni_in * 4;
  const size_t nd_out = JW;                                         // prio
  const size_t ni_out = W + JW + 2 + J + J + (J + 1) + (size_t)totw + 2 * (size_t)J + (size_t)totw;
  const size_t out_bytes = nd_out * 8 + ni_out * 4 + J;
  std::vector<unsigned char> h(in_bytes);
  double *hd = reinterpret_cast<double *>(h.data());
  memcpy(hd, a->alloc, JW * 8); memcpy(hd + JW, a->job_time, JW * 8); memcpy(hd + 2 * JW, a->thr, JW * 8);
  memcpy(hd + 3 * JW, a->deficit, JW * 8); memcpy(hd + 4 * JW, a->worker_time, (size_t)W * 8);
  int32_t *hi = reinterpret_cast<int32_t *>(hd + nd_in);
  size_t o = 0;
  auto put = [&](const int32_t *src, size_t n) { memcpy(hi + o, src, n * 4); size_t at = o; o += n; return at; };
  const size_t o_order = put(a->type_order, W), o_cap = put(a->capacity, W), o_sf = put(a->sf, J),
               o_nw = put(a->nworkers, W), o_wid = put(a->worker_ids, totw), o_pt = put(a->prev_type, J),
               o_po = put(a->prev_off, J + 1), o_pl = put(a->prev_local, nprev);
  CK(c->gv_out.need(out_bytes, c->st));
  CK(c->gv_in.upload(h.data(), in_bytes, c->st));
  const double *dd = c->gv_in.as<double>();
  const int32_t *di = reinterpret_cast<const int32_t *>(dd + nd_in);
  double *od = c->gv_out.as<double>();
  int32_t *oi = reinterpret_cast<int32_t *>(od + nd_out);
  swb::GavelLaunch L;
  L.J = J; L.W = W; L.flags = a->flags; L.maxw = maxw;
  L.alloc = dd; L.job_time = dd + JW; L.thr = dd + 2 * JW; L.deficit = dd + 3 * JW; L.worker_time = dd + 4 * JW;
  L.type_order = di + o_order; L.capacity = di + o_cap; L.sf = di + o_sf; L.nworkers = di + o_nw;
  L.worker_ids = di + o_wid; L.prev_type = di + o_pt; L.prev_off = di + o_po; L.prev_local = di + o_pl;
  L.in_alloc = nullptr;
  L.prio = od;
  size_t q = 0;
  L.n_sel = oi + q; q += W;
  L.sel_jobs = oi + q; q += JW;
  L.out_scalars = oi + q; q += 2;
  L.assign_job = oi + q; q += J;
  L.assign_cnt = oi + q; q += J;
  L.assign_off = oi + q; q += J + 1;
  L.assign_workers = oi + q; q += totw;
  L.tmp_rank0 = oi + q; q += J;
  q += J;
  L.tmp_free = oi + q; q += totw;
  L.sched = reinterpret_cast<uint8_t *>(oi + ni_out);
  CK(swb::launch_gavel_round(L, c->st));
  std::vector<unsigned char> ho(out_bytes);
  CK(cudaMemcpyAsync(ho.data(), c->gv_out.p, out_bytes, cudaMemcpyDeviceToHost, c->st));
  CK(cudaStreamSynchronize(c->st));
  const double *rd = reinterpret_cast<const double *>(ho.data());
  const int32_t *ri = reinterpret_cast<const int32_t *>(rd + nd_out);
  memcpy(a->prio, rd, JW * 8);
  memcpy(a->n_sel, ri, (size_t)W * 4);
  memcpy(a->sel_jobs, ri + W, JW * 4);
  const int32_t nasg = ri[W + JW], err = ri[W + JW + 1];
  *a->n_assigned = nasg;
  memcpy(a->assign_job, ri + W + JW + 2, (size_t)J * 4);
  memcpy(a->assign_off, ri + W + JW + 2 + 2 * (size_t)J, (size_t)(J + 1) * 4);
  memcpy(a->assign_workers, ri + W + JW + 2 + 2 * (size_t)J + (J + 1), (size_t)totw * 4);
  if (err) return fail(SWB_ERR_STATE, "swb_gavel_round: could not assign workers to a selected job (scheduler.py:1097-1100)");
  return 0;
}

int swb_gbm_ensemble(swb_ctx *c, int32_t S, int32_t J, double P_total, const double *sums_dev, const double *z,
                     double *rem_out_dev) {
  if (!c || !sums_dev || !z || !rem_out_dev) return fail(SWB_ERR_ARG, "swb_gbm_ensemble: null argument");
  if (S <= 0 || J <= 0 || !(P_total > 0.0)) return fail(SWB_ERR_ARG, "swb_gbm_ensemble: bad S / J / P_total");
  CK(cudaSetDevice(c->device));
  CK(c->ens_z.upload(z, (size_t)S * 8, c->st));
  CK(swb::launch_gbm_ensemble(S, J, P_total, sums_dev, c->ens_z.as<double>(), rem_out_dev, c->st));
  if (!c->aux_async) CK(cudaStreamSynchronize(c->st));
  return 0;
}

// One level of the market iteration: measurement pass, start pass, `iters` x (dense step + dual step).  Events around
// the last dense step when `timed`.
static int market_level(swb_ctx *c, swb::MarketLaunch &L, int iters, bool timed) {
  const size_t nwt = (size_t)L.S * L.W * L.T;
  CK(swb::launch_market_fill(L.colscale, nwt, 1.0f, c->st));
  CK(swb::launch_market_fill(L.pws, (size_t)L.S, L.pw, c->st));
  CK(cudaMemsetAsync(L.colload, 0, nwt * 4, c->st));
  CK(cudaMemsetAsync(L.rowp, 0, (size_t)L.S * L.J * 4, c->st));
  L.phase = 0;                                           // per-job constants (jobpack) for the measurement pass
  CK(swb::launch_market_iter(L, c->st, false));
  L.mode = 1;                                            // measurement: X clamped to [0,1], reductions filled
  CK(swb::launch_market_iter(L, c->st, true));
  CK(swb::launch_market_iter(L, c->st, false));          // start: reductions of x^0 remembered, theta / prices from the duals
  L.mode = 0; L.phase = 1;
  for (int it = 0; it < iters; ++it) {
    const int slot = it - (iters - swb_ctx::MEV / 2);      // the last MEV/2 dense passes are timed one by one
    if (timed && slot >= 0) CK(cudaEventRecord(c->mev[2 * slot], c->st));
    CK(swb::launch_market_iter(L, c->st, true));
    if (timed && slot >= 0) CK(cudaEventRecord(c->mev[2 * slot + 1], c->st));
    CK(swb::launch_market_iter(L, c->st, false));
  }
  return 0;
}

int swb_market_pgd(swb_ctx *c, const swb_market_args *a) {
  if (!c || !a || !a->prm || !a->g || !a->E || !a->c || !a->dbar || !a->rem || !a->rate || (!a->Gw && !a->cap) || !a->X)
    return fail(SWB_ERR_ARG, "swb_market_pgd: null argument");
  const int S = a->S, J = a->J, W = a->W, T = a->T;
  if (S <= 0 || J <= 0 || W <= 0 || W > SWB_MK_MAXW || T <= 0 || (T & 3) || T > 1024)
    return fail(SWB_ERR_ARG, "swb_market_pgd: need W in [1,4], T a multiple of 4, T <= 1024");
  if (a->iters < 0 || a->coarse_iters < 0 || a->primal_weight < 0.f)
    return fail(SWB_ERR_ARG, "swb_market_pgd: negative iteration count or primal weight");
  const int TC = 4, grp = T / TC;
  const bool coarse = a->coarse_iters > 0 && T >= 16;
  // 1 / capacity per (type, round), fine and coarse (mean over the group of rounds), host side: W T numbers
  std::vector<float> icap((size_t)W * T + (size_t)W * TC);
  for (int w = 0; w < W; ++w) {
    for (int t = 0; t < T; ++t) {
      const double cv = a->cap ? a->cap[(size_t)w * T + t] : a->Gw[w];
      if (!(cv > 0.0)) return fail(SWB_ERR_ARG, "swb_market_pgd: capacities must be positive");
      icap[(size_t)w * T + t] = (float)(1.0 / cv);
    }
    for (int tc = 0; tc < TC; ++tc) {
      double m = 0.0;
      for (int t = tc * grp; t < (tc + 1) * grp; ++t) m += a->cap ? a->cap[(size_t)w * T + t] : a->Gw[w];
      icap[(size_t)W * T + (size_t)w * TC + tc] = (float)((double)grp / m);
    }
  }
  CK(cudaSetDevice(c->device));
  const size_t nj = a->per_scenario_jobs ? (size_t)S * J : (size_t)J, sj = (size_t)S * J;
  const size_t nx = sj * W * T, nwt = (size_t)S * W * T, nwc = (size_t)S * W * TC;
  CK(c->prm.upload(a->prm, sizeof(swb_params) * S, c->st));
  CK(c->m_theta.need(sj * 16, c->st)); CK(c->m_rowp.need(sj * 4, c->st));
  CK(c->m_rowprev.need(sj * 4, c->st)); CK(c->m_mj.need(sj * 8, c->st)); CK(c->m_om.need(sj * 8, c->st));
  CK(c->m_colload.need(nwt * 4, c->st)); CK(c->m_colscale.need(nwt * 4, c->st)); CK(c->m_price.need(nwt * 4, c->st));
  CK(c->m_colprev.need(nwt * 4, c->st)); CK(c->m_pi.need(nwt * 8, c->st));
  CK(c->m_obj.need((size_t)S * 3 * 8, c->st));
  CK(c->m_Gw.upload(icap.data(), icap.size() * 4, c->st));
  swb::MarketLaunch L;
  L.S = S; L.J = J; L.W = W; L.T = T; L.per_scn = a->per_scenario_jobs;
  L.Tfull = T; L.rscale = 1.f;
  L.prm = c->prm.as<swb_params>(); L.icap = c->m_Gw.as<float>();
  if (a->on_device) {
    L.g = a->g; L.E = a->E; L.c = a->c; L.dbar = a->dbar; L.rem = a->rem; L.rate = a->rate; L.X = a->X;
  } else {
    CK(c->g.upload(a->g, nj * 4, c->st));
    CK(c->m_E.upload(a->E, nj * 8, c->st));
    CK(c->m_c.upload(a->c, nj * 8, c->st));
    CK(c->dbar.upload(a->dbar, nj * 8, c->st));
    CK(c->rem.upload(a->rem, nj * 8, c->st));
    CK(c->m_rate.upload(a->rate, nj * W * 4, c->st));
    CK(c->m_X.need(nx * 4, c->st));
    if (a->warm_start) CK(cudaMemcpyAsync(c->m_X.p, a->X, nx * 4, cudaMemcpyHostToDevice, c->st));
    L.g = c->g.as<int32_t>(); L.E = c->m_E.as<double>(); L.c = c->m_c.as<double>();
    L.dbar = c->dbar.as<double>(); L.rem = c->rem.as<double>(); L.rate = c->m_rate.as<float>();
    L.X = c->m_X.as<float>();
  }
  if (!a->warm_start) CK(cudaMemsetAsync(L.X, 0, nx * 4, c->st));
  L.jobpack = c->m_theta.as<float4>();
  L.rowp = c->m_rowp.as<float>(); L.rowprev = c->m_rowprev.as<float>();
  L.mj = c->m_mj.as<double>(); L.om = c->m_om.as<double>();
  L.colload = c->m_colload.as<float>(); L.colprev = c->m_colprev.as<float>();
  L.colscale = c->m_colscale.as<float>(); L.price = c->m_price.as<float>(); L.pi = c->m_pi.as<double>();
  L.obj = c->m_obj.as<double>();
  if (a->utility != 0 && a->utility != 1) return fail(SWB_ERR_ARG, "swb_market_pgd: utility must be 0 or 1");
  L.utility = a->utility;
  const double pwrel = a->primal_weight > 0.f ? (double)a->primal_weight : (a->utility == 1 ? 1.0 : 60.0);
  L.pw = (float)(pwrel / ((double)J * (double)T));
  CK(c->m_pws.need((size_t)S * 4, c->st));
  L.pws = c->m_pws.as<float>();
  L.phase = 0; L.mode = 0;
  const int split = 8;                 // CTAs per scenario (8 sweeps per thread at 4096 jobs x 64 rounds)
  auto tile = [&](int Tl) {            // jobs per CTA: enough CTAs to fill the GPU, long sweeps so the column accumulators pay
    int per = (J + split - 1) / split;
    const int sweep = 256 / (Tl / 4) > 0 ? 256 / (Tl / 4) : 1;
    per = ((per + sweep - 1) / sweep) * sweep;
    return per < sweep ? sweep : per;
  };
  // duals start at zero: marginal utilities, makespan multipliers, prices
  CK(cudaMemsetAsync(L.mj, 0, sj * 8, c->st)); CK(cudaMemsetAsync(L.om, 0, sj * 8, c->st));
  CK(cudaMemsetAsync(L.pi, 0, nwt * 8, c->st));
  if (coarse) {
    // level 1: the same iteration on X_c[S][J][W][4] — one entry stands for T/4 rounds (rate x T/4, mean capacity)
    CK(c->m_Xc.need(sj * W * TC * 4, c->st));
    CK(c->m_cc.need(nwc * (4 * 4 + 8), c->st));
    swb::MarketLaunch Lc = L;
    Lc.T = TC; Lc.rscale = (float)grp; Lc.X = c->m_Xc.as<float>(); Lc.icap = L.icap + (size_t)W * T;
    float *cc = c->m_cc.as<float>();
    Lc.colload = cc; Lc.colprev = cc + nwc; Lc.colscale = cc + 2 * nwc; Lc.price = cc + 3 * nwc;
    Lc.pi = reinterpret_cast<double *>(cc + 4 * nwc);
    Lc.jobs_per_cta = tile(TC);
    CK(cudaMemsetAsync(Lc.pi, 0, nwc * 8, c->st));
    if (a->warm_start) CK(swb::launch_market_restrict(L.X, Lc.X, sj * W, T, grp, c->st));
    else CK(cudaMemsetAsync(Lc.X, 0, sj * W * TC * 4, c->st));
    if (int rc = market_level(c, Lc, a->coarse_iters, false)) return rc;
    CK(swb::launch_market_prolong(Lc.X, L.X, Lc.pi, L.pi, sj * W, S, W, T, grp, c->st));
  }
  L.jobs_per_cta = tile(T);
  if (int rc = market_level(c, L, a->iters, true)) return rc;
  // objective and violation of the last iterate, then make it feasible (column scaling) and score that
  float dense_ms = 0.f;
  L.phase = 2;
  CK(swb::launch_market_iter(L, c->st, false));
  L.mode = 1;
  CK(swb::launch_market_iter(L, c->st, true));
  L.phase = 3;
  CK(swb::launch_market_iter(L, c->st, false));
  if (a->obj) CK(cudaMemcpyAsync(a->obj, L.obj, (size_t)S * 3 * 8, cudaMemcpyDeviceToHost, c->st));
  if (!a->on_device) CK(cudaMemcpyAsync(a->X, L.X, nx * 4, cudaMemcpyDeviceToHost, c->st));
  CK(cudaStreamSynchronize(c->st));
  {
    // mean over the timed passes (the event clock of some boxes ticks in coarse steps: one pass alone reads as a
    // multiple of the tick)
    const int first = a->iters >= swb_ctx::MEV / 2 ? 0 : swb_ctx::MEV / 2 - a->iters;
    int n = 0;
    double acc = 0.0;
    for (int sl = first; sl < swb_ctx::MEV / 2 && a->iters > 0; ++sl) {
      float ms = 0.f;
      CK(cudaEventElapsedTime(&ms, c->mev[2 * sl], c->mev[2 * sl + 1]));
      acc += ms; ++n;
    }
    dense_ms = n ? (float)(acc / n) : 0.f;
  }
  if (a->dense_ms) *a->dense_ms = dense_ms;
  return 0;
}

int swb_set_option(swb_ctx *c, int32_t option, int32_t value) {
  if (!c) return fail(SWB_ERR_ARG, "null ctx");
  if (option == SWB_OPT_RELAXED_OPTIMUM) { c->want_relaxed = value ? 1 : 0; return 0; }
  if (option == SWB_OPT_SOLVE_CLUSTER) { c->solve_cluster = (value == 8) ? 8 : 1; return 0; }
  if (option == SWB_OPT_ASYNC_AUX) { c->aux_async = value ? 1 : 0; return 0; }
  if (option == SWB_OPT_RERANK_ITERS) { c->rr_iters = value < 0 ? 0 : value; return 0; }
  if (option == SWB_OPT_RERANK_RESTARTS) { c->rr_restarts = value < 0 ? 0 : (value > 16 ? 16 : value); return 0; }
  if (option == SWB_OPT_GBM_PATHS) { if (value < 0) return fail(SWB_ERR_ARG, "paths < 0"); c->gbm_paths = value; return 0; }
  if (option == SWB_OPT_GBM_SEED) { c->gbm_seed = (uint64_t)(uint32_t)value; return 0; }
  if (option == SWB_OPT_GBM_HORIZON) { if (value < 1) return fail(SWB_ERR_ARG, "horizon < 1"); c->gbm_hmax = value; return 0; }
  return fail(SWB_ERR_ARG, "swb_set_option: unknown option");
}

int swb_allox_assign(swb_ctx *c, int32_t m, int32_t n, int32_t W, const double *p, const double *t,
                     const int32_t *wtype, int32_t *col_of_job, double *total_cost) {
  if (!c || !p || !t || !wtype || !col_of_job) return fail(SWB_ERR_ARG, "swb_allox_assign: null argument");
  if (m <= 0 || n <= 0 || W <= 0 || (long long)m * n > (1ll << 26))
    return fail(SWB_ERR_ARG, "swb_allox_assign: need m, n > 0 and m*n <= 2^26");
  CK(cudaSetDevice(c->device));
  const size_t N = (size_t)m * n;
  CK(c->ax_u.need((size_t)m * 8, c->st));
  CK(c->ax_v.need(N * 8, c->st)); CK(c->ax_spc.need(N * 8, c->st));
  CK(c->ax_c4r.need((size_t)m * 4, c->st)); CK(c->ax_r4c.need(N * 4, c->st)); CK(c->ax_path.need(N * 4, c->st));
  CK(c->ax_sc.need(N, c->st)); CK(c->ax_sr.need((size_t)m, c->st)); CK(c->ax_out.need(8, c->st));
  CK(c->ax_p.upload(p, (size_t)m * W * 8, c->st));
  CK(c->ax_t.upload(t, (size_t)m * 8, c->st));
  CK(c->ax_wt.upload(wtype, (size_t)n * 4, c->st));
  swb::AssignLaunch L;
  L.m = m; L.n = n; L.W = W;
  L.p = c->ax_p.as<double>(); L.t = c->ax_t.as<double>(); L.wtype = c->ax_wt.as<int32_t>();
  L.u = c->ax_u.as<double>(); L.v = c->ax_v.as<double>(); L.spc = c->ax_spc.as<double>();
  L.col4row = c->ax_c4r.as<int32_t>(); L.row4col = c->ax_r4c.as<int32_t>(); L.path = c->ax_path.as<int32_t>();
  L.inSC = c->ax_sc.as<unsigned char>(); L.inSR = c->ax_sr.as<unsigned char>(); L.out = c->ax_out.as<double>();
  CK(swb::launch_assign(L, c->st));
  double tot = 0.0;
  CK(cudaMemcpyAsync(col_of_job, L.col4row, (size_t)m * 4, cudaMemcpyDeviceToHost, c->st));
  CK(cudaMemcpyAsync(&tot, L.out, 8, cudaMemcpyDeviceToHost, c->st));
  CK(cudaStreamSynchronize(c->st));
  if (total_cost) *total_cost = tot;
  return 0;
}

int swb_lp_solve(swb_ctx *c, int32_t S, int32_t m, int32_t n, int32_t nnz, const int32_t *colp, const int32_t *rowi,
                 const double *val, const double *cost, const double *b, int32_t max_iter, double *x,
                 double *objective, int32_t *status, int32_t *stats) {
  if (!c || !colp || !rowi || !val || !cost || !b || !x || !objective || !status)
    return fail(SWB_ERR_ARG, "swb_lp_solve: null argument");
  if (S <= 0 || S > 4096 || m <= 0 || m > 2048 || n <= 0 || n > (1 << 22) || nnz < 0 || max_iter <= 0)
    return fail(SWB_ERR_ARG, "swb_lp_solve: need 1 <= S <= 4096, 1 <= m <= 2048, 1 <= n <= 2^22, max_iter > 0");
  if ((size_t)S * m * m * 16 > ((size_t)8 << 30))
    return fail(SWB_ERR_ARG, "swb_lp_solve: S * m^2 * 16 bytes of basis inverses exceed 8 GiB");
  if (colp[0] != 0 || colp[n] != nnz) return fail(SWB_ERR_ARG, "swb_lp_solve: colp[0] must be 0 and colp[n] == nnz");
  for (int j = 0; j < n; ++j)
    if (colp[j + 1] < colp[j]) return fail(SWB_ERR_ARG, "swb_lp_solve: colp must be non-decreasing");
  for (int k = 0; k < nnz; ++k)
    if (rowi[k] < 0 || rowi[k] >= m) return fail(SWB_ERR_ARG, "swb_lp_solve: row index out of range");
  CK(cudaSetDevice(c->device));
  const size_t sm = (size_t)S * m, sn = (size_t)S * n, snz = (size_t)S * (nnz > 0 ? nnz : 1);
  CK(c->lp_rowi.need((size_t)(nnz > 0 ? nnz : 1) * 4, c->st)); CK(c->lp_val.need(snz * 8, c->st));
  CK(c->lp_Binv.need(sm * m * 8, c->st)); CK(c->lp_Bm.need(sm * m * 8, c->st)); CK(c->lp_vec.need(sm * 5 * 8, c->st));
  CK(c->lp_basis.need(sm * 4, c->st)); CK(c->lp_where.need((size_t)S * (n + m + 1) * 4, c->st));
  CK(c->lp_x.need(sn * 8, c->st)); CK(c->lp_out.need((size_t)S * 64, c->st));
  CK(c->lp_colp.upload(colp, (size_t)(n + 1) * 4, c->st));
  if (nnz > 0) {
    CK(cudaMemcpyAsync(c->lp_rowi.p, rowi, (size_t)nnz * 4, cudaMemcpyHostToDevice, c->st));
    CK(cudaMemcpyAsync(c->lp_val.p, val, (size_t)S * nnz * 8, cudaMemcpyHostToDevice, c->st));
  }
  CK(c->lp_c.upload(cost, sn * 8, c->st));
  CK(c->lp_b.upload(b, sm * 8, c->st));
  swb::LpLaunch L;
  L.S = S; L.m = m; L.n = n; L.nnz = nnz; L.max_iter = max_iter;
  L.colp = c->lp_colp.as<int>(); L.rowi = c->lp_rowi.as<int>();
  L.val = c->lp_val.as<double>(); L.c = c->lp_c.as<double>(); L.b = c->lp_b.as<double>();
  L.Binv = c->lp_Binv.as<double>(); L.Bm = c->lp_Bm.as<double>(); L.vec = c->lp_vec.as<double>();
  L.basis = c->lp_basis.as<int>(); L.where = c->lp_where.as<int>();
  L.x = c->lp_x.as<double>(); L.out = c->lp_out.as<double>();
  CK(swb::launch_lp(L, c->st));
  std::vector<double> out((size_t)S * 8);
  CK(cudaMemcpyAsync(x, c->lp_x.p, sn * 8, cudaMemcpyDeviceToHost, c->st));
  CK(cudaMemcpyAsync(out.data(), c->lp_out.p, (size_t)S * 64, cudaMemcpyDeviceToHost, c->st));
  CK(cudaStreamSynchronize(c->st));
  int worst = 0;
  for (int s = 0; s < S; ++s) {
    objective[s] = out[(size_t)s * 8];
    status[s] = (int32_t)out[(size_t)s * 8 + 1];
    if (status[s] > worst) worst = status[s];
    if (stats)
      for (int k = 0; k < 4; ++k) stats[s * 4 + k] = (int32_t)out[(size_t)s * 8 + 2 + k];
  }
  return worst >= 3 ? fail(SWB_ERR_STATE, "swb_lp_solve: a program hit the pivot limit or a singular basis (see status[])") : 0;
}

int swb_last_timings(swb_ctx *c, double *ms_solve, double *ms_place, int32_t *passes) {
  if (!c) return fail(SWB_ERR_ARG, "null ctx");
  float a = 0.f, b = 0.f;
  CK(cudaEventElapsedTime(&a, c->ev[0], c->ev[1]));
  CK(cudaEventElapsedTime(&b, c->ev[1], c->ev[2]));
  if (ms_solve) *ms_solve = a;
  if (ms_place) *ms_place = b;
  if (passes) *passes = c->last_passes;
  return 0;
}

int swb_forecast_commit(swb_ctx *c, int32_t J, int32_t fallback, const int32_t *ncal) {
  if (!c || !ncal) return fail(SWB_ERR_ARG, "swb_forecast_commit: null argument");
  if (!c->have_fc || c->last_fc.J != J) return fail(SWB_ERR_STATE, "swb_forecast_commit: no matching forecast");
  CK(cudaSetDevice(c->device));
  CK(c->f_ncal.upload(ncal, (size_t)J * 4, c->st));
  CK(swb::launch_commit_calibration(c->last_fc, nullptr, fallback, c->f_ncal.as<int32_t>(), c->st));
  CK(cudaStreamSynchronize(c->st));
  c->have_fc = false;
  return 0;
}

}  // extern "C"
