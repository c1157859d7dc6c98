// place.cu — dense J x T placement of the solved round counts, objective re-evaluation on the
// placed schedule, and the work-conserving back-fill.
//
// Reference behaviour replaced:
//   * the x[j][t] values Gurobi returns for a given set of per-job counts (any permutation of rounds
//     is equally optimal for the MILP, SURVEY.md §0 R3) — here a deterministic water-filling packer:
//     jobs in descending width take their n_j least-loaded rounds, rounds then ordered by planned work;
//   * rank_in_schedule_jobs() (scheduler/shockwave.py:714-793), the second MILP of the fallback
//     path: minimise sum_j prio_j * mean round index with the counts fixed — here a priority round-sweep
//     keyed by prio_j / (n_j g_j) (the exchange-argument order for that linear objective) over the leading
//     rounds, and the water-filling packer with rounds ordered by sum prio_j/n_j for what the sweep leaves;
//   * construct_schedules() (shockwave.py:213-285): per round, idle GPUs are back-filled with the
//     not-yet-scheduled jobs in descending remaining-runtime order (stable) that still fit.
//
// One CTA per scenario.  Round masks (128 bit per job) live in shared memory for J <= 4096.
// G must fit 24 bits (bin keys are load<<8|bin).
#include <math.h>

#include "swb_common.cuh"
#include "swb_internal.h"
#include "rerank.cuh"
#include <cooperative_groups.h>

namespace swb {

// bitonic sort, DESCENDING by (key, then ascending idx) over n = power of two entries (n >= 64, blockDim a multiple of
// 32).  Strides >= 32 go through shared memory (one barrier each); the strides 16..1 that end every merge level stay in
// registers: element i lives in lane i % 32 of its warp, its partner i ^ j in lane (i % 32) ^ j, so the five
// compare-exchanges are shuffles with one barrier for all of them (36 barriers instead of 78 at n = 4096).
__device__ void sort_desc64(unsigned long long *key, unsigned short *idx, int n) {
  for (int k = 2; k <= n; k <<= 1) {
    // all levels k <= 32 run inside one register pass (k = 32 carries them)
    if (k < 32) continue;
    int j = k >> 1;
    for (; j >= 32; j >>= 1) {
      for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const int p = i ^ j;
        if (p > i) {
          const unsigned long long a = key[i], b = key[p];
          const unsigned short ia = idx[i], ib = idx[p];
          const bool a_first = (a > b) || (a == b && ia < ib);  // a belongs before b
          const bool up = (i & k) == 0;
          if (up != a_first) { key[i] = b; key[p] = a; idx[i] = ib; idx[p] = ia; }
        }
      }
      __syncthreads();
    }
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
      unsigned long long a = key[i];
      int ia = idx[i];
      for (int kk = (k == 32 ? 2 : k); kk <= k; kk <<= 1) {
        const bool up = (i & kk) == 0;
        for (int jj = (kk >> 1) > 16 ? 16 : (kk >> 1); jj > 0; jj >>= 1) {
          const unsigned long long b = __shfl_xor_sync(SWB_FULL, a, jj);
          const int ib = __shfl_xor_sync(SWB_FULL, ia, jj);
          const bool mine_first = (a > b) || (a == b && ia < ib);
          const bool keep_first = (((i & jj) == 0) == up);
          if (keep_first != mine_first) { a = b; ia = ib; }
        }
      }
      key[i] = a;
      idx[i] = (unsigned short)ia;
    }
    __syncthreads();
  }
}


__host__ __device__ __forceinline__ int sort_pad(int J) {   // sort length: a power of two >= max(J, 64)
  int npad = 64;
  while (npad < J) npad <<= 1;
  return npad;
}

// Dynamic shared memory of one placement CTA.  The per-round arrays hold SWB_MAX_T entries, the per-job ones npad.
struct PlaceSmem {
  double *red;                   // BlockRed scratch
  int *idle, *load_of;           // idle GPUs per round; load of every bin the packer filled
  unsigned int *binA, *binB;     // the packer's bins, load << 8 | bin, sorted by load (two buffers)
  double *score;                 // planned work of every bin
  unsigned char *newpos;         // bin -> its rank among the packer's rounds
  ulonglong2 *pmask;             // prefix OR of the bin bits behind the ring's physical positions [0, q) (chunk path)
  unsigned long long *key64;     // sort scratch: key64[npad] + idx16[npad]
  unsigned short *idx16;
  unsigned short *rank;          // job -> position in the priority order
  unsigned short *order;         // jobs in back-fill order
  unsigned char *gs, *remn;      // width; rounds still to seat (the plan until the job is seated)
  unsigned char *ext;            // rounds added by the improvement pass beyond the plan
  unsigned char *remr;           // remaining counts of the priority round-sweep (fallback re-rank)
  unsigned short *ordr;          // jobs by priority density
  unsigned long long *xm, *bm;   // [J][2] each: round masks of the schedule and the back-fill (null: J > SWB_SMEM_JOBS)
  unsigned char *rr_hot;         // hot arrays of the re-rank search (w_j, dense edge costs), null unless `hot`
};

// Carves the dynamic shared memory at `base` (16-byte aligned) and returns its size; with base = nullptr it only
// sizes.  The round masks follow the sort scratch up to SWB_SMEM_JOBS jobs, and with `hot` the search's hot arrays
// follow the masks.
__host__ __device__ __forceinline__ size_t place_carve(PlaceSmem &m, unsigned char *base, int J, int T, bool hot) {
  const size_t npad = (size_t)sort_pad(J);
  unsigned char *p = base;
  m.red = reinterpret_cast<double *>(p);             p += 2 * 64 * sizeof(double);
  m.idle = reinterpret_cast<int *>(p);               p += SWB_MAX_T * sizeof(int);
  m.load_of = reinterpret_cast<int *>(p);            p += SWB_MAX_T * sizeof(int);
  m.binA = reinterpret_cast<unsigned int *>(p);      p += SWB_MAX_T * sizeof(int);
  m.binB = reinterpret_cast<unsigned int *>(p);      p += SWB_MAX_T * sizeof(int);
  m.score = reinterpret_cast<double *>(p);           p += SWB_MAX_T * sizeof(double);
  m.newpos = p;                                      p += SWB_MAX_T;
  m.pmask = reinterpret_cast<ulonglong2 *>(p);       p += (SWB_MAX_T + 1) * sizeof(ulonglong2);
  m.key64 = reinterpret_cast<unsigned long long *>(p);
  m.idx16 = reinterpret_cast<unsigned short *>(p + 8 * npad);
  p += 10 * npad;
  m.rank = reinterpret_cast<unsigned short *>(p);    p += 2 * npad;
  m.order = reinterpret_cast<unsigned short *>(p);   p += 2 * npad;
  m.gs = p;   p += npad;
  m.remn = p; p += npad;
  m.ext = p;  p += npad;
  m.remr = p; p += npad;
  m.ordr = reinterpret_cast<unsigned short *>(p);    p += 2 * npad;
  p = align16(p);
  m.xm = m.bm = nullptr;
  m.rr_hot = nullptr;
  if (J <= SWB_SMEM_JOBS) {
    m.xm = reinterpret_cast<unsigned long long *>(p); p += 16 * (size_t)J;
    m.bm = reinterpret_cast<unsigned long long *>(p); p += 16 * (size_t)J;
    if (hot) {
      RrScratch r;
      rr_carve(r, nullptr, nullptr, J, T);
      m.rr_hot = p; p += r.hot_bytes;
    }
  }
  return (size_t)(p - base);
}

// What the phases of one scenario's placement share.
struct PlaceCta {
  PlaceSmem m;
  BlockRed br;
  int s, J, T, G, npad;
  size_t so;                 // first row of the scenario in the [S][J] arrays
  bool fallback;             // the solve fell back: priority order, sweep and re-rank search (with L.weights)
  bool prio;                 // fallback && L.weights
  const uint8_t *nplan;      // planned round counts
  int t0;                    // rounds [0, t0) are seated by the sweep (bits kept in bm until merged into xm)
  int Tw;                    // rounds the water-filling packer works on ("bins" 0..Tw-1 = rounds t0..T-1)

  __device__ __forceinline__ PlaceCta(const PlaceLaunch &L, int s_, unsigned char *smem, unsigned long long *gmask)
      : br(nullptr), s(s_), J(L.J) {
    T = L.prm[s].future_rounds; G = L.prm[s].ngpus;
    so = (size_t)s * J;
    npad = sort_pad(J);
    place_carve(m, smem, J, T, L.plan.hot_smem != 0);
    if (J > SWB_SMEM_JOBS) {
      m.xm = gmask + (size_t)s * 4 * J;
      m.bm = m.xm + 2 * (size_t)J;
    }
    br = BlockRed(m.red);
    fallback = (L.res[s].status == SWB_ST_FALLBACK);
    prio = fallback && L.weights;
    nplan = L.sc_n + so;
    t0 = 0; Tw = T;
  }
};

// CTA -> scenario: longest first.  A fallback scenario costs about twice a plain one here (priority sweep), and with
// two waves of CTAs the launch ends when the slowest SM finishes: CTA b takes the b-th fallback scenario while
// there are any, then the plain ones (the result does not depend on the mapping).
__device__ __forceinline__ int cta_scenario(const PlaceLaunch &L, int b, int *s_scan, int *s_scn) {
  const int chunk = (L.S + (int)blockDim.x - 1) / (int)blockDim.x;
  const int c0 = min(L.S, (int)threadIdx.x * chunk), c1 = min(L.S, c0 + chunk);
  int cnt = 0;
  for (int i = c0; i < c1; ++i) cnt += (L.res[i].status == SWB_ST_FALLBACK) ? 1 : 0;
  int tot = 0;
  const int pre = block_excl_scan(cnt, s_scan, &tot);
  const bool want_fb = b < tot;
  const int target = want_fb ? b : b - tot;
  const int mypre = want_fb ? pre : (c0 - pre);
  const int mycnt = want_fb ? cnt : (c1 - c0 - cnt);
  if (target >= mypre && target < mypre + mycnt) {
    int seen = mypre;
    for (int i = c0; i < c1; ++i) {
      const bool fb = (L.res[i].status == SWB_ST_FALLBACK);
      if (fb == want_fb) { if (seen == target) { *s_scn = i; break; } ++seen; }
    }
  }
  __syncthreads();
  return *s_scn;
}

// Fallback packing order: higher prio_j/(n_j g_j) first, the exchange-argument order of rank_in_schedule_jobs.
// Fills rank (job -> position) and ordr (position -> job, 0xffff: padding).
__device__ __forceinline__ void priority_order(const PlaceCta &c, const PlaceLaunch &L) {
  const PlaceSmem &m = c.m;
  const int J = c.J, npad = c.npad;
  const double *wj = L.weights + c.so;
  for (int i = threadIdx.x; i < npad; i += blockDim.x) {
    double d = -1.0;
    if (i < J && c.nplan[i] > 0) d = wj[i] / ((double)c.nplan[i] * (double)m.gs[i]);
    m.key64[i] = (i < J) ? order_key(d) : 0ull;
    m.idx16[i] = (unsigned short)(i < J ? i : 0xffff);
  }
  __syncthreads();
  sort_desc64(m.key64, m.idx16, npad);
  for (int i = threadIdx.x; i < npad; i += blockDim.x) {
    if (m.idx16[i] != 0xffff) m.rank[m.idx16[i]] = (unsigned short)i;
    m.ordr[i] = m.idx16[i];
  }
  __syncthreads();
}

// One round of the sweep, part (b): a SEQUENTIAL greedy in priority order — a job is seated if it still fits — walked
// by warp 0 alone, 128 jobs per step (4 per lane): no block barrier inside the walk (the block-wide multi-pass form of
// this loop spent ~16 barriers per round and dominated the fallback placement at 4096 jobs).  The greedy is the fixed
// point of "take the longest prefix of the eligible jobs that fits, repeat", i.e. exactly what that form computed.
// blk_min[b] = a lower bound of the narrowest job of block b (128 consecutive jobs of the priority order) that still
// needs rounds — refreshed whenever the walk visits the block, stale only on the low side (jobs finish, they never
// come back) — so a block whose bound exceeds the capacity left is skipped without being read; a round that ends with
// a few idle GPUs nobody fits costs two ballots, not a scan.  Returns the capacity left.
__device__ __forceinline__ int sweep_walk(const PlaceCta &c, const unsigned char *g_o, unsigned char *rem_o,
                                          const unsigned char *flag_o, unsigned short *blk_min, int cap, int t) {
  const int lane = threadIdx.x, npad = c.npad;
  const int wt = t >> 6;
  const unsigned long long bt = 1ull << (t & 63);
  const unsigned char mark = (unsigned char)(t + 1);
  const int nblk = (npad + 127) >> 7;     // <= 64
  int nextb = 0;
  while (cap > 0) {
    const unsigned int m0 = __ballot_sync(SWB_FULL, lane < nblk && (int)blk_min[lane] <= cap);
    const unsigned int m1 = __ballot_sync(SWB_FULL, lane + 32 < nblk && (int)blk_min[lane + 32] <= cap);
    unsigned long long mm = ((unsigned long long)m1 << 32) | m0;
    mm &= (nextb >= 64) ? 0ull : (~0ull << nextb);
    if (mm == 0ull) break;
    const int blk = __ffsll((long long)mm) - 1;
    nextb = blk + 1;
    const int q0 = (blk << 7) + 4 * lane;
    int g[4], rem[4];
    bool el[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const bool in = q0 + e < npad;
      g[e] = in ? (int)g_o[q0 + e] : 0; rem[e] = in ? (int)rem_o[q0 + e] : 0;
      el[e] = rem[e] > 0 && flag_o[in ? q0 + e : 0] != mark && g[e] <= cap;
    }
    while (true) {
      int inc[4], sloc = 0;
#pragma unroll
      for (int e = 0; e < 4; ++e) { if (el[e]) sloc += g[e]; inc[e] = sloc; }
      if (!__any_sync(SWB_FULL, sloc > 0)) break;
      int incl = sloc;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(SWB_FULL, incl, o); if (lane >= o) incl += v; }
      const int excl = incl - sloc;
      int got = 0, vpos = 128;
#pragma unroll
      for (int e = 3; e >= 0; --e) {
        if (el[e]) {
          if (excl + inc[e] <= cap) {
            got += g[e];
            rem[e] -= 1; rem_o[q0 + e] = (unsigned char)rem[e];
            c.m.bm[2 * c.m.ordr[q0 + e] + wt] |= bt;
            el[e] = false;
          } else {
            vpos = 4 * lane + e;           // ends as this lane's FIRST job that did not fit
          }
        }
      }
      got = __reduce_add_sync(SWB_FULL, got);
      vpos = __reduce_min_sync(SWB_FULL, vpos);
      cap -= got;
      if (vpos == 128) break;
#pragma unroll
      for (int e = 0; e < 4; ++e) el[e] = el[e] && (4 * lane + e) > vpos && g[e] <= cap;
    }
    int lm = 0xffff;
#pragma unroll
    for (int e = 0; e < 4; ++e) if (rem[e] > 0) lm = min(lm, g[e]);
    lm = __reduce_min_sync(SWB_FULL, lm);
    if (lane == 0) blk_min[blk] = (unsigned short)lm;
    __syncwarp();
  }
  return cap;
}

// Fallback re-rank (rank_in_schedule_jobs, shockwave.py:714-793): minimise sum_j prio_j * mean round index with the
// counts fixed.  Round-by-round priority sweep: a round first seats the jobs that can no longer wait (remaining count
// == rounds left), then the jobs of highest prio_j/(n_j g_j) that still fit — for unit widths this greedy is optimal by
// an exchange argument and always feasible (McNaughton).  With mixed widths a round can fragment.  The sweep therefore
// stops at the first round t0 after which the remaining counts provably no longer pack (GPU-rounds left > G * rounds
// left, or the jobs that need every remaining round are wider than the cluster), takes that round back, and hands the
// remaining counts over rounds [t0, T) to the water-filling packer (which packs whenever the width classes nest, and
// orders its rounds by priority score).  Sets c.t0, remr and remn.
__device__ __forceinline__ void priority_sweep(PlaceCta &c) {
  const PlaceSmem &m = c.m;
  const int J = c.J, T = c.T, G = c.G, npad = c.npad;
  const uint8_t *nplan = c.nplan;
  const int chs = (npad + blockDim.x - 1) / blockDim.x;
  const int p0 = threadIdx.x * chs;
  long long dem = 0;     // GPU-rounds still to seat; they must fit the rounds that remain
  for (int j = threadIdx.x; j < J; j += blockDim.x) dem += (long long)m.gs[j] * nplan[j];
  dem = c.br.sumll(dem);
  // the sweep works on arrays IN PRIORITY ORDER (contiguous, one 32-bit word = 4 consecutive jobs; the sort scratch is
  // free here): width, remaining count, "seated in round t" marker (t + 1)
  unsigned char *g_o = reinterpret_cast<unsigned char *>(m.key64), *rem_o = g_o + npad, *flag_o = g_o + 2 * (size_t)npad;
  for (int pos = threadIdx.x; pos < npad; pos += blockDim.x) {
    const int j = m.ordr[pos];
    const bool v = (j != 0xffff);
    g_o[pos] = v ? m.gs[j] : 0; rem_o[pos] = v ? nplan[j] : 0; flag_o[pos] = 0;
  }
  __syncthreads();
  c.t0 = T;
  // One round = (a) the CRITICAL jobs (remaining count == rounds left; all of them must fit) seated by the whole block
  // with one reduction, then (b) the greedy walk of warp 0 (sweep_walk).
  __shared__ int s_sw_cap;
  __shared__ unsigned short blk_min[64];              // 0xffff: nobody in the block needs rounds any more
  if (threadIdx.x < 64) blk_min[threadIdx.x] = 0;     // 0 = unknown: visit
  int fail = 0, tfail = 0;
  for (int t = 0; t < T; ++t) {
    const int tau = T - t;
    int capleft = G;
    const int wt = t >> 6;
    const unsigned long long bt = 1ull << (t & 63);
    const unsigned char mark = (unsigned char)(t + 1);
    // (a) critical jobs
    int csum = 0;
    for (int q = 0; q < chs; ++q) {
      const int pos = p0 + q;
      if (pos < npad && rem_o[pos] > 0 && rem_o[pos] >= tau) csum += g_o[pos];
    }
    const int ctot = (int)c.br.sumll((long long)csum);
    if (ctot > capleft) {
      fail = 1;                                  // the critical jobs alone do not fit
    } else {
      if (csum > 0)
        for (int q = 0; q < chs; ++q) {
          const int pos = p0 + q;
          if (pos < npad && rem_o[pos] > 0 && rem_o[pos] >= tau) {
            m.bm[2 * m.ordr[pos] + wt] |= bt; rem_o[pos] = (unsigned char)(rem_o[pos] - 1); flag_o[pos] = mark;
          }
        }
      capleft -= ctot;
      __syncthreads();
      // (b) greedy walk by warp 0
      if (threadIdx.x < 32) {
        const int cap = sweep_walk(c, g_o, rem_o, flag_o, blk_min, capleft, t);
        if (threadIdx.x == 0) s_sw_cap = cap;
      }
      __syncthreads();
      const int ncap = s_sw_cap;
      dem -= (long long)(G - ncap);
      capleft = ncap;
    }
    if (!fail) {
      if (threadIdx.x == 0) m.idle[t] = capleft;
      if (dem > (long long)G * (tau - 1)) fail = 2;   // what is left no longer fits the rounds that remain
    }
    if (fail) { tfail = t; break; }
  }
  __syncthreads();
  for (int pos = threadIdx.x; pos < npad; pos += blockDim.x) {
    const int j = m.ordr[pos];
    if (j != 0xffff) m.remr[j] = rem_o[pos];
  }
  __syncthreads();
  if (fail) {
    // fail 1 is detected before round t seats anybody: the culprit is round t-1; fail 2: round t itself
    const int tr = (fail == 1 && tfail > 0) ? tfail - 1 : tfail;
    for (int j = threadIdx.x; j < J; j += blockDim.x) {
      const unsigned long long bit = 1ull << (tr & 63);
      if (m.bm[2 * j + (tr >> 6)] & bit) { m.bm[2 * j + (tr >> 6)] &= ~bit; m.remr[j] = (unsigned char)(m.remr[j] + 1); }
    }
    c.t0 = tr;
  }
  __syncthreads();
  for (int j = threadIdx.x; j < J; j += blockDim.x) m.remn[j] = m.remr[j];
  __syncthreads();
}

// Chunk-parallel path of the water-filling walk: 32 consecutive jobs of the SAME width on a balanced ring.
// With the bins sorted by load and max - min <= g, least-loaded-first over jobs of width g is a round-robin over the
// ring: job i takes the ring positions [head + P_i, head + P_i + n_i) (P = exclusive prefix sum of the counts), the
// order stays sorted and the spread stays <= g.  The bin behind every ring position does not change, so the 32 jobs
// compute their round masks independently; only the fit (no bin above G at the END of the chunk) has to be checked
// first.  The result is identical to seating the 32 jobs one after the other.  Returns false (nothing seated) when the
// chunk does not qualify; else pos is the chunk's last job.
__device__ __forceinline__ bool seat_chunk(const PlaceCta &c, int lane, unsigned int *A, int &pos, int &head,
                                           bool &pm_ok) {
  const PlaceSmem &m = c.m;
  const int J = c.J, G = c.G, Tw = c.Tw;
  const int pp = pos + lane;
  const bool valid0 = pp < J && m.key64[pp] != 0ull;
  const int jj = valid0 ? (int)m.idx16[pp] : 0;
  const int gg0 = valid0 ? (int)m.gs[jj] : 0;
  const int g0 = __shfl_sync(SWB_FULL, gg0, 0);
  // the chunk = the leading run of jobs of the first job's width (at a boundary between two width classes the
  // run is shorter than 32; the next iteration starts on the new width)
  const unsigned int okm = __ballot_sync(SWB_FULL, valid0 && gg0 == g0);
  const int cnt = (okm == 0xffffffffu) ? 32 : (__ffs((int)~okm) - 1);
  const bool valid = lane < cnt;
  const int nn = valid ? (int)m.remn[jj] : 0;
  int hl0 = head + Tw - 1; if (hl0 >= Tw) hl0 -= Tw;
  const int lmin = (int)(A[head] >> 8), lmax = (int)(A[hl0] >> 8);
  int incl = nn;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { const int t2 = __shfl_up_sync(SWB_FULL, incl, o); if (lane >= o) incl += t2; }
  const int Ptot = __shfl_sync(SWB_FULL, incl, 31);
  const int cfull = Ptot / Tw, rpart = Ptot - cfull * Tw;
  int hr = head + rpart - 1; if (hr >= Tw) hr -= Tw; if (hr < 0) hr += Tw;
  const int top = max(rpart > 0 ? (int)(A[hr] >> 8) + g0 * (cfull + 1) : 0, lmax + g0 * cfull);
  const bool short_ok = __all_sync(SWB_FULL, nn <= Tw);
  if (!(cnt >= 4 && short_ok && lmax - lmin <= g0 && top <= G)) return false;
  if (!pm_ok) {
    // the bins behind a ring range [a, b) as a mask = pmask[b] ^ pmask[a] (every bin appears once): one warp
    // scan here replaces a dependent walk over up to T shared-memory reads per job
    unsigned long long c0 = 0ull, c1 = 0ull, l0[4], l1[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int pq = 4 * lane + e;
      if (pq < Tw) {
        const unsigned int b = A[pq] & 0xffu;
        if (b < 64) c0 |= 1ull << b; else c1 |= 1ull << (b - 64);
      }
      l0[e] = c0; l1[e] = c1;
    }
    unsigned long long i0 = c0, i1 = c1;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned long long t0_ = __shfl_up_sync(SWB_FULL, i0, o), t1_ = __shfl_up_sync(SWB_FULL, i1, o);
      if (lane >= o) { i0 |= t0_; i1 |= t1_; }
    }
    unsigned long long e0 = __shfl_up_sync(SWB_FULL, i0, 1), e1 = __shfl_up_sync(SWB_FULL, i1, 1);
    if (lane == 0) { e0 = 0ull; e1 = 0ull; m.pmask[0] = make_ulonglong2(0ull, 0ull); }
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int pq = 4 * lane + e;
      if (pq < Tw) m.pmask[pq + 1] = make_ulonglong2(e0 | l0[e], e1 | l1[e]);
    }
    pm_ok = true;
    __syncwarp();
  }
  if (valid) {
    int st = head + (incl - nn) % Tw; if (st >= Tw) st -= Tw;
    const int en = st + nn;
    const ulonglong2 pa = m.pmask[st];
    unsigned long long m0, m1;
    if (en <= Tw) {
      const ulonglong2 pb = m.pmask[en];
      m0 = pb.x ^ pa.x; m1 = pb.y ^ pa.y;
    } else {
      const ulonglong2 pe = m.pmask[Tw], pb = m.pmask[en - Tw];
      m0 = (pe.x ^ pa.x) | pb.x; m1 = (pe.y ^ pa.y) | pb.y;
    }
    m.xm[2 * jj] = m0; m.xm[2 * jj + 1] = m1; m.remn[jj] = 0;
  }
  __syncwarp();
  for (int p = lane; p < Tw; p += 32) {           // loads after the whole chunk
    int off = p - head; if (off < 0) off += Tw;
    A[p] += (unsigned)(g0 * (cfull + (off < rpart ? 1 : 0))) << 8;
  }
  head += rpart; if (head >= Tw) head -= Tw;
  pos += cnt - 1;
  __syncwarp();
  return true;
}

// Water-filling, run by warp 0 on the jobs sorted by packing_keys: each job takes its n_j least-loaded rounds ("bins")
// that still fit it.  With widths in descending order the loads stay multiples of the current width, so there is no
// fragmentation; least-loaded-first keeps the loads level.  One warp walks the jobs; the bins are kept sorted by
// (load, bin) and re-merged after every job.
__device__ __forceinline__ void waterfill_walk(const PlaceCta &c) {
  const PlaceSmem &m = c.m;
  const int J = c.J, G = c.G, Tw = c.Tw;
  const int lane = threadIdx.x;
  unsigned int *A = m.binA, *B = m.binB;
  for (int p = lane; p < Tw; p += 32) A[p] = (unsigned)p;  // load 0, bin p
  __syncwarp();
  int head = 0;   // the sorted bins are a RING: logical position p lives in A[(head + p) mod Tw]
  bool pm_ok = false;   // pmask[] matches the current physical order of A
  for (int pos = 0; pos < J; ++pos) {
    if (m.key64[pos] == 0ull) break;
    if (seat_chunk(c, lane, A, pos, head, pm_ok)) continue;
    const int j = m.idx16[pos];
    // remn == plan until the job is seated (shared memory; nplan is global).  Only lane 0 touches remn[] on this
    // path (it also writes it below), the count reaches the other lanes by shuffle.
    const int g = m.gs[j], n = __shfl_sync(SWB_FULL, lane == 0 ? (int)m.remn[j] : 0, 0);
    const unsigned int lim = ((unsigned)(G - g) << 8) | 0xffu;
    const unsigned int add = (unsigned)g << 8;
    // Fast path (the common, load-balanced state): the n least-loaded bins all fit the job and, once
    // raised by g, are at least as loaded as the currently most loaded bin -> moving them to the END
    // of the order keeps it sorted by load; in a ring that is just `head += n`, no data moves.
    // (Ties between equal loads are broken by age instead of bin id; any least-loaded choice is valid.)
    int hn = head + n - 1; if (hn >= Tw) hn -= Tw;
    int hl = head + Tw - 1; if (hl >= Tw) hl -= Tw;
    const unsigned int vn = A[hn], vl = A[hl], v0 = A[head];
    // every moved bin must end up at least as loaded as the most loaded unmoved one: test the SMALLEST
    if (vn <= lim && (v0 >> 8) + (unsigned)g >= (vl >> 8)) {
      unsigned int w0 = 0, w1 = 0, w2 = 0, w3 = 0;
      for (int p = lane; p < n; p += 32) {
        int ix = head + p; if (ix >= Tw) ix -= Tw;
        const unsigned int v = A[ix];
        A[ix] = v + add;
        const unsigned int b = v & 0xffu;
        const unsigned int bit = 1u << (b & 31);
        if (b < 32) w0 |= bit; else if (b < 64) w1 |= bit; else if (b < 96) w2 |= bit; else w3 |= bit;
      }
      w0 = __reduce_or_sync(SWB_FULL, w0); w1 = __reduce_or_sync(SWB_FULL, w1);
      w2 = __reduce_or_sync(SWB_FULL, w2); w3 = __reduce_or_sync(SWB_FULL, w3);
      if (lane == 0) {
        m.xm[2 * j] = (unsigned long long)w0 | ((unsigned long long)w1 << 32);
        m.xm[2 * j + 1] = (unsigned long long)w2 | ((unsigned long long)w3 << 32);
        m.remn[j] = 0;
      }
      head += n; if (head >= Tw) head -= Tw;
      __syncwarp();
      continue;
    }
    // General path: linearise the ring, then take the usable prefix and re-merge.
    pm_ok = false;
    if (head != 0) {
      for (int p = lane; p < Tw; p += 32) { int ix = head + p; if (ix >= Tw) ix -= Tw; B[p] = A[ix]; }
      unsigned int *tmp0 = A; A = B; B = tmp0;
      head = 0;
      __syncwarp();
    }
    int u = 0;
    for (int p = lane; p < Tw; p += 32) u += (A[p] <= lim) ? 1 : 0;
    u = warp_sum(u);
    const int mm = n < u ? n : u;
    if (mm > 0) {
      unsigned long long m0 = 0ull, m1 = 0ull;
      for (int p = lane; p < mm; p += 32) {
        const unsigned int b = A[p] & 0xffu;
        if (b < 64) m0 |= 1ull << b; else m1 |= 1ull << (b - 64);
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        m0 |= __shfl_xor_sync(SWB_FULL, m0, o);
        m1 |= __shfl_xor_sync(SWB_FULL, m1, o);
      }
      if (lane == 0) { m.xm[2 * j] = m0; m.xm[2 * j + 1] = m1; m.remn[j] = (unsigned char)(n - mm); }
      if (mm == Tw) {
        for (int p = lane; p < Tw; p += 32) A[p] += add;
      } else {
        // stable merge BY LOAD of X = A[0..mm)+add with Y = A[mm..Tw): equal loads keep the unmoved bins
        // first (both runs are sorted by load; the bin id in the low byte is not part of the order)
        for (int p = lane; p < Tw; p += 32) {
          int dst;
          if (p < mm) {
            const unsigned int v = A[p] + add, lv = v >> 8;
            int lo = mm, hi = Tw;               // #{y in Y : load(y) <= load(v)}
            while (lo < hi) { const int mid = (lo + hi) >> 1; if ((A[mid] >> 8) <= lv) lo = mid + 1; else hi = mid; }
            dst = p + (lo - mm);
            B[dst] = v;
          } else {
            const unsigned int v = A[p], lv = v >> 8;
            int lo = 0, hi = mm;               // #{x in X : load(x) < load(v)}
            while (lo < hi) { const int mid = (lo + hi) >> 1; if (((A[mid] + add) >> 8) < lv) lo = mid + 1; else hi = mid; }
            dst = (p - mm) + lo;
            B[dst] = v;
          }
        }
        unsigned int *tmp = A; A = B; B = tmp;
      }
      __syncwarp();
    }
  }
  // the bins' loads for the round order (order_rounds); scores start at zero
  for (int p = lane; p < Tw; p += 32) { m.load_of[A[p] & 0xffu] = (int)(A[p] >> 8); m.score[p] = 0.0; }
}

// The water-filling packer over rounds [t0, T): sort the jobs with counts left (packing_keys), then warp 0 walks them.
__device__ __forceinline__ void waterfill(const PlaceCta &c) {
  const PlaceSmem &m = c.m;
  const int J = c.J, npad = c.npad;
  for (int i = threadIdx.x; i < npad; i += blockDim.x) {
    unsigned long long k = 0ull;
    if (i < J && m.remn[i] > 0) {
      // jobs that need (almost) every round must come first inside their width class or the rounds
      // they need fill up; the fallback priority only breaks ties (it drives the round ORDER below)
      const unsigned long long tie = c.prio ? (unsigned long long)(SWB_MAX_J - m.rank[i])
                                            : (unsigned long long)(SWB_MAX_J - 1 - i);
      // a job present in EVERY round only lowers all capacities by g: seat those first, whatever
      // their width — a narrow all-rounds job seated late finds some rounds already full
      const unsigned long long all_rounds = ((int)m.remn[i] >= c.Tw) ? 1ull : 0ull;
      k = (all_rounds << 48) | ((unsigned long long)m.gs[i] << 40) | ((unsigned long long)m.remn[i] << 28) |
          (tie << 14) | (unsigned long long)(SWB_MAX_J - 1 - i);
    }
    m.key64[i] = k;
    m.idx16[i] = (unsigned short)(i < J ? i : 0xffff);
  }
  __syncthreads();
  sort_desc64(m.key64, m.idx16, npad);
  if (threadIdx.x < 32) waterfill_walk(c);
}

// Packing order: wider gangs first, then more planned rounds (fallback: higher prio_j/(n_j g_j)), then job index.
// The remainder of a partial sweep can fail to pack although the full plan does (the sweep spent the narrow jobs
// early).  Then the sweep is shortened — to 3/4, 1/2, 1/4 of its rounds, then none — and the packer runs again.
__device__ __forceinline__ void pack(PlaceCta &c) {
  const PlaceSmem &m = c.m;
  const int J = c.J;
  const int t0_sweep = c.t0;
  for (int att = 0;; ++att) {
    c.Tw = c.T - c.t0;
    if (c.Tw > 0) waterfill(c);
    __syncthreads();
    if (c.t0 == 0) break;
    long long sf = 0;
    for (int j = threadIdx.x; j < J; j += blockDim.x) sf += m.remn[j];
    sf = c.br.sumll(sf);
    if (sf == 0) break;
    const int nt0 = att < 3 ? (t0_sweep * (3 - att)) / 4 : 0;
    // give back the sweep's rounds [nt0, t0): their bits leave bm, their counts return to the packer
    for (int j = threadIdx.x; j < J; j += blockDim.x) {
      int back = 0;
      for (int wi = 0; wi < 2; ++wi) {
        const int lo = max(nt0 - 64 * wi, 0), hi = min(c.t0 - 64 * wi, 64);
        if (hi > lo) {
          const unsigned long long mk = ((hi >= 64) ? ~0ull : ((1ull << hi) - 1ull)) & ~((1ull << lo) - 1ull);
          back += __popcll(m.bm[2 * j + wi] & mk);
          m.bm[2 * j + wi] &= ~mk;
        }
      }
      m.remr[j] = (unsigned char)(m.remr[j] + back);
      m.remn[j] = m.remr[j];
      m.xm[2 * j] = 0; m.xm[2 * j + 1] = 0;
    }
    c.t0 = nt0;
    __syncthreads();
  }
}

// Order the packer's rounds: interchangeable for the MILP objective, so put first the rounds that carry the most
// planned work (fallback: the largest sum of prio_j/n_j, which minimises sum_j prio_j * mean round index for this
// partition — rearrangement inequality).  Then move every job's bins to their rounds and merge the sweep's rounds.
__device__ __forceinline__ void order_rounds(const PlaceCta &c, const PlaceLaunch &L) {
  const PlaceSmem &m = c.m;
  const int J = c.J, Tw = c.Tw, t0 = c.t0;
  if (Tw > 0) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    for (int b = warp; b < Tw; b += nw) {
      double acc = 0.0;
      for (int j = lane; j < J; j += 32) {
        if ((m.xm[2 * j + (b >> 6)] >> (b & 63)) & 1ull)
          acc += c.prio ? L.weights[c.so + j] / (double)c.nplan[j] : (double)c.nplan[j] * (double)m.gs[j];
      }
      acc = warp_sum(acc);
      if (lane == 0) m.score[b] = acc;
    }
    __syncthreads();
    for (int b = threadIdx.x; b < Tw; b += blockDim.x) {
      const double sb = m.score[b];
      int r = 0;
      for (int o = 0; o < Tw; ++o) { const double so2 = m.score[o]; r += (so2 > sb || (so2 == sb && o < b)) ? 1 : 0; }
      m.newpos[b] = (unsigned char)r;
      m.idle[t0 + r] = c.G - m.load_of[b];
    }
    __syncthreads();
  }
  for (int j = threadIdx.x; j < J; j += blockDim.x) {
    unsigned long long o0 = 0ull, o1 = 0ull;
    for (int wi = 0; wi < 2; ++wi) {
      unsigned long long mm = m.xm[2 * j + wi];
      while (mm) {
        const int b = __ffsll((long long)mm) - 1; mm &= mm - 1;
        const int t = t0 + m.newpos[64 * wi + b];
        if (t < 64) o0 |= 1ull << t; else o1 |= 1ull << (t - 64);
      }
    }
    m.xm[2 * j] = o0 | m.bm[2 * j]; m.xm[2 * j + 1] = o1 | m.bm[2 * j + 1];   // + the rounds seated by the sweep
    m.bm[2 * j] = 0; m.bm[2 * j + 1] = 0;
  }
  __syncthreads();
}

// Fallback re-rank, second stage: negative-cycle cancelling on the round graph (rerank.cuh) improves the sweep's
// schedule towards the optimum of rank_in_schedule_jobs (shockwave.py:714-793); only when every planned round was
// seated and the plan admits the search (plan_place).  With a cluster, all CTAs of the scenario search from different
// seeds and the one with the best schedule carries on alone.  Returns false in the CTAs that are done; *rr_cycles =
// cycles cancelled (| winning start << 12).
template <int CL>
__device__ __forceinline__ bool rerank(PlaceCta &c, const PlaceLaunch &L, int crank, int *rr_cycles) {
  namespace cg = cooperative_groups;
  const PlaceSmem &m = c.m;
  const int J = c.J;
  if (c.prio && L.plan.rerank) {
    long long sfl = 0;
    for (int j = threadIdx.x; j < J; j += blockDim.x) sfl += m.remn[j];
    sfl = c.br.sumll(sfl);
    __shared__ double s_rr_cost;
    if (threadIdx.x == 0) s_rr_cost = 1e300;
    __syncthreads();
    if (sfl == 0) {
      *rr_cycles = rr_local_search(reinterpret_cast<unsigned char *>(L.rr_items) +
                                       ((size_t)c.s * CL + crank) * L.plan.rr_region, m.rr_hot,
                                   m.xm, m.gs, m.remn, c.nplan, L.weights + c.so, m.idle, J, c.T, L.rr_iters,
                                   crank == 0 ? 0u : (unsigned)(crank * 7919 + 13), L.rr_restarts, &s_rr_cost);
      __syncthreads();
    }
    if constexpr (CL > 1) {
      // best of the cluster's 8 searches carries on; the others are done (two barriers: nobody leaves while its
      // cost may still be read)
      cg::cluster_group cl = cg::this_cluster();
      cl.sync();
      int win = 0;
      double bestc = *cl.map_shared_rank(&s_rr_cost, 0);
      for (int r = 1; r < CL; ++r) {
        const double cr = *cl.map_shared_rank(&s_rr_cost, r);
        if (cr < bestc) { bestc = cr; win = r; }
      }
      cl.sync();
      if (crank != win) return false;
      *rr_cycles |= win << 12;          // reported in swb_result.flags: which start won
    }
  } else {
    if constexpr (CL > 1) { if (crank != 0) return false; }
  }
  return true;
}

// Improvement pass: GPU-rounds the packing left idle go to the job with the best marginal utility per GPU that is not
// yet in that round and still fits (only matters when the counts could not be packed perfectly: wide gangs on a small
// cluster).
__device__ __forceinline__ void improve(PlaceCta &c, const PlaceLaunch &L, const Pwl &P) {
  const PlaceSmem &m = c.m;
  const int J = c.J, T = c.T;
  const size_t so = c.so;
  const uint8_t *nplan = c.nplan;
  int any = 0;
  for (int j = threadIdx.x; j < J; j += blockDim.x)
    any |= ((int)nplan[j] - (int)m.remn[j] < (int)L.sc_nmax[so + j]) ? 1 : 0;
  any = (int)c.br.sumll((long long)any);
  int idle_tot = 0;
  for (int t = 0; t < T; ++t) idle_tot += m.idle[t];
  if (any && idle_tot > 0) {
    const double Dd = L.prm[c.s].round_duration;
    int budget = 64;
    for (int t = 0; t < T && budget > 0; ++t) {
      while (m.idle[t] > 0 && budget > 0) {
        const int room = m.idle[t];
        double bd = 0.0;
        for (int j = threadIdx.x; j < J; j += blockDim.x) {
          const int n = (int)nplan[j] - (int)m.remn[j] + (int)m.ext[j];
          if (n < (int)L.sc_nmax[so + j] && (int)m.gs[j] <= room && !((m.xm[2 * j + (t >> 6)] >> (t & 63)) & 1ull)) {
            const double a = L.sc_a[so + j], u0 = L.sc_u0[so + j], cap = L.sc_cap[so + j];
            const double u1 = util_u(a, u0, cap, Dd, n + 1), u_0 = util_u(a, u0, cap, Dd, n);
            bd = fmax(bd, L.sc_ws[so + j] * (plog(P, u1) - plog(P, u_0)) / (double)m.gs[j]);
          }
        }
        bd = c.br.max(bd);
        if (!(bd > 0.0)) break;
        double bj = 1e300;
        for (int j = threadIdx.x; j < J; j += blockDim.x) {
          const int n = (int)nplan[j] - (int)m.remn[j] + (int)m.ext[j];
          if (n < (int)L.sc_nmax[so + j] && (int)m.gs[j] <= room && !((m.xm[2 * j + (t >> 6)] >> (t & 63)) & 1ull)) {
            const double a = L.sc_a[so + j], u0 = L.sc_u0[so + j], cap = L.sc_cap[so + j];
            const double u1 = util_u(a, u0, cap, Dd, n + 1), u_0 = util_u(a, u0, cap, Dd, n);
            if (L.sc_ws[so + j] * (plog(P, u1) - plog(P, u_0)) / (double)m.gs[j] >= bd) bj = fmin(bj, (double)j);
          }
        }
        bj = c.br.min(bj);
        if (bj >= 1e299) break;
        const int wj = (int)bj;
        if (threadIdx.x == 0) {
          m.xm[2 * wj + (t >> 6)] |= 1ull << (t & 63);
          m.ext[wj] = (unsigned char)(m.ext[wj] + 1);
          m.idle[t] = room - (int)m.gs[wj];
        }
        --budget;
        __syncthreads();
      }
    }
  }
  __syncthreads();
}

// Objective of the PLACED schedule (what a checker recomputes from x) into the scenario's result; also the round counts
// and the unscheduled rounds with idle GPUs per job.  Returns the rounds left unseated, *me_all = the makespan term.
__device__ __forceinline__ long long objective(PlaceCta &c, const PlaceLaunch &L, const Pwl &P, int rr_cycles,
                                               double *me_all) {
  const PlaceSmem &m = c.m;
  const int J = c.J, T = c.T;
  const size_t so = c.so;
  const swb_params &prm = L.prm[c.s];
  double w = 0.0, me = 0.0;
  long long shortf = 0;
  for (int j = threadIdx.x; j < J; j += blockDim.x) {
    const int n = (int)c.nplan[j] - (int)m.remn[j] + (int)m.ext[j];
    shortf += m.remn[j];
    // same float64 formula a checker applies to x: p = min(D n / dbar, E - c), u = (c + p) / E
    const size_t ji = (L.per_scn ? so : 0) + j;
    const double Ef = (double)L.E[ji], cf = (double)L.c[ji], db = L.dbar[ji];
    const double pj = fmin(prm.round_duration * (double)n / db, Ef - cf);
    w += L.sc_ws[so + j] * plog(P, (cf + pj) / Ef);
    const double done = db * pj;
    me = fmax(me, fmax(0.0, L.sc_R[so + j] - done));
    if (L.nrounds) L.nrounds[so + j] = n;
    if (L.ncal) {
      int mc = 0;
      for (int t = 0; t < T; ++t)
        mc += (m.idle[t] > 0 && !((m.xm[2 * j + (t >> 6)] >> (t & 63)) & 1ull)) ? 1 : 0;
      L.ncal[so + j] = mc;
    }
  }
  w = c.br.sum(w);
  me = c.br.max(me);
  shortf = c.br.sumll(shortf);
  *me_all = me;
  if (threadIdx.x == 0) {
    swb_result &r = L.res[c.s];
    r.welfare = w; r.makespan = me; r.objective = w - prm.k * me; r.shortfall = (int)shortf;
    r.placement = c.t0;
    r.flags = (r.flags & 0xff) | (rr_cycles << 8);      // cycles cancelled by the re-rank local search
  }
  return shortf;
}

// Packing feedback for the next pass (api.cu re-solves while rounds stay unseated).
// The price-based counts only know the aggregate capacity G*T; when gang widths do not nest in G (one 8-gang per
// 12-GPU round) a width class can be over-planned and the packer strands whoever comes last in its order.  Which
// job-rounds of that class to give up is an economic choice, not a packing one: for every stranded job-round, the job
// of the SAME width whose last planned round is worth least (welfare slope + makespan term) loses one round via ncap;
// the next solve re-prices everything else around the tighter class.
__device__ __forceinline__ void packing_feedback(PlaceCta &c, const PlaceLaunch &L, const Pwl &P, double me_all,
                                                 long long shortf_all) {
  const PlaceSmem &m = c.m;
  const int J = c.J;
  const size_t so = c.so;
  const swb_params &prm = L.prm[c.s];
  unsigned char *cuts = m.remr, *covered = m.ext;       // both arrays are free at this point
  for (int j = threadIdx.x; j < J; j += blockDim.x) { cuts[j] = 0; covered[j] = 0; }
  __syncthreads();
  const double Dd = prm.round_duration;
  const int budget = shortf_all < 96 ? (int)shortf_all : 96;
  for (int it = 0; it < budget; ++it) {
    double fk = -1.0;                                // stranded job: widest first, then lowest index
    for (int j = threadIdx.x; j < J; j += blockDim.x)
      if ((int)m.remn[j] > (int)covered[j]) fk = fmax(fk, (double)m.gs[j] * 16384.0 + (double)(SWB_MAX_J - 1 - j));
    fk = c.br.max(fk);
    if (fk < 0.0) break;
    const int gf = (int)(fk / 16384.0);
    const int f = SWB_MAX_J - 1 - (int)(fk - (double)gf * 16384.0);
    double bl = 1e300;
    for (int pass2 = 0; pass2 < 2; ++pass2) {
      double v = 1e300;
      for (int j = threadIdx.x; j < J; j += blockDim.x) {
        const int n = (int)c.nplan[j] - (int)cuts[j];
        if ((int)m.gs[j] != gf || n < 1) continue;
        const double a = L.sc_a[so + j], u0 = L.sc_u0[so + j], cap = L.sc_cap[so + j];
        const double u1 = util_u(a, u0, cap, Dd, n), u_0 = util_u(a, u0, cap, Dd, n - 1);
        const size_t ji = (L.per_scn ? so : 0) + j;
        const double db = L.dbar[ji], room = (double)L.E[ji] - (double)L.c[ji];
        const double rem0 = fmax(0.0, L.sc_R[so + j] - db * fmin(Dd * (double)(n - 1) / db, room));
        const double loss = L.sc_ws[so + j] * (plog(P, u1) - plog(P, u_0)) + prm.k * fmax(0.0, rem0 - me_all);
        if (pass2 == 0) v = fmin(v, loss);
        else if (loss <= bl) v = fmin(v, (double)j);
      }
      bl = c.br.min(v);                              // second pass: bl = index of the cheapest round
    }
    if (bl >= 1e299) break;
    if (threadIdx.x == 0) { cuts[(int)bl] = (unsigned char)(cuts[(int)bl] + 1); covered[f] = (unsigned char)(covered[f] + 1); }
    __syncthreads();
  }
  for (int j = threadIdx.x; j < J; j += blockDim.x)
    if (cuts[j] > 0) {
      const int capn = (int)c.nplan[j] - (int)cuts[j];
      if (capn < (int)L.ncap[so + j]) L.ncap[so + j] = (uint8_t)capn;
    }
  __syncthreads();
}

// Work-conserving back-fill: one warp per round walks the sorted order (descending remaining runtime, stable,
// shockwave.py:261-267).  The order costs a full sort of the jobs and is only needed when some round has idle GPUs
// left; a window whose rounds are all full skips it.
__device__ __forceinline__ void backfill(const PlaceCta &c, const PlaceLaunch &L) {
  const PlaceSmem &m = c.m;
  const int J = c.J, T = c.T, npad = c.npad;
  int any_idle = 0;
  for (int t = threadIdx.x; t < T; t += blockDim.x) any_idle |= m.idle[t] > 0 ? 1 : 0;
  any_idle = __syncthreads_or(any_idle);
  if (!any_idle) return;
  const double *bk = ((c.fallback && L.bfkey_fb) ? L.bfkey_fb : L.bfkey) + (L.per_scn ? c.so : 0);
  for (int i = threadIdx.x; i < npad; i += blockDim.x) {
    m.key64[i] = (i < J) ? order_key(bk[i]) : 0ull;
    m.idx16[i] = (unsigned short)(i < J ? i : 0xffff);
  }
  __syncthreads();
  sort_desc64(m.key64, m.idx16, npad);
  for (int i = threadIdx.x; i < npad; i += blockDim.x) m.order[i] = m.idx16[i];
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  for (int t = warp; t < T; t += nw) {
    int left = m.idle[t];
    const int wi = t >> 6;
    const unsigned long long bit = 1ull << (t & 63);
    for (int base = 0; base < J && left > 0; base += 32) {
      const int pos = base + lane;
      int j = -1, g = 0;
      if (pos < J) {
        j = m.order[pos];
        g = m.gs[j];
        if (m.xm[2 * j + wi] & bit) j = -1;
      }
      unsigned int mb = __ballot_sync(SWB_FULL, j >= 0 && g <= left);
      while (mb && left > 0) {
        const int l = __ffs(mb) - 1;
        mb &= mb - 1;
        const int gl = __shfl_sync(SWB_FULL, g, l);
        if (gl <= left) {
          left -= gl;
          if (lane == l) atomicOr(&m.bm[2 * j + wi], bit);
        }
      }
    }
  }
}

// Outputs: 128-bit round masks (16 B per job and matrix) and/or byte matrices, coalesced.
__device__ __forceinline__ void write_outputs(const PlaceCta &c, const PlaceLaunch &L) {
  const PlaceSmem &m = c.m;
  const int J = c.J, T = c.T;
  const size_t so = c.so;
  if (L.xmask || L.bfmask) {
    for (int e = threadIdx.x; e < 2 * J; e += blockDim.x) {
      if (L.xmask) L.xmask[2 * so + e] = m.xm[e];
      if (L.bfmask) L.bfmask[2 * so + e] = m.bm[e];
    }
  }
  const size_t xo = so * (size_t)T;
  if ((T & 3) == 0) {
    const int total4 = J * (T >> 2), q4 = T >> 2;
    unsigned int *x4 = reinterpret_cast<unsigned int *>(L.x ? L.x + xo : nullptr);
    unsigned int *b4 = reinterpret_cast<unsigned int *>(L.backfill ? L.backfill + xo : nullptr);
    for (int e = threadIdx.x; e < total4; e += blockDim.x) {
      const int j = e / q4, t = (e - j * q4) << 2;
      const int sh = t & 63, wi = t >> 6;
      if (x4) {
        const unsigned int mk = (unsigned int)(m.xm[2 * j + wi] >> sh) & 0xfu;
        x4[e] = (mk & 1u) | ((mk & 2u) << 7) | ((mk & 4u) << 14) | ((mk & 8u) << 21);
      }
      if (b4) {
        const unsigned int mk = (unsigned int)(m.bm[2 * j + wi] >> sh) & 0xfu;
        b4[e] = (mk & 1u) | ((mk & 2u) << 7) | ((mk & 4u) << 14) | ((mk & 8u) << 21);
      }
    }
  } else {
    const int total = J * T;
    for (int e = threadIdx.x; e < total; e += blockDim.x) {
      const int j = e / T, t = e - j * T;
      const int wi = t >> 6;
      const unsigned long long bit = 1ull << (t & 63);
      if (L.x) L.x[xo + e] = (m.xm[2 * j + wi] & bit) ? 1 : 0;
      if (L.backfill) L.backfill[xo + e] = (m.bm[2 * j + wi] & bit) ? 1 : 0;
    }
  }
}

// CL = 1: one CTA per scenario.  CL = 8 (few scenarios, the re-rank search on): a thread-block cluster per scenario —
// all 8 CTAs build the same schedule, each runs the re-rank local search from a different noising seed (rank 0: none),
// the costs meet through distributed shared memory and the CTA with the best schedule carries on alone.
template <int CL>
__global__ void __launch_bounds__(SWB_PLACE_THREADS, 1) place_kernel(PlaceLaunch L, unsigned long long *gmask) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  int crank = 0;
  if constexpr (CL > 1) crank = (int)cooperative_groups::this_cluster().block_rank();
  __shared__ int s_scan[33], s_scn;
  PlaceCta c(L, cta_scenario(L, blockIdx.x / CL, s_scan, &s_scn), smem_raw, gmask);
  for (int j = threadIdx.x; j < c.J; j += blockDim.x) {
    c.m.gs[j] = L.sc_g[c.so + j]; c.m.remn[j] = c.nplan[j]; c.m.ext[j] = 0;
    c.m.xm[2 * j] = 0; c.m.xm[2 * j + 1] = 0; c.m.bm[2 * j] = 0; c.m.bm[2 * j + 1] = 0;
  }
  __syncthreads();
  if (c.prio) {
    priority_order(c, L);
    priority_sweep(c);
  }
  pack(c);
  order_rounds(c, L);
  int rr_cycles = 0;
  if (!rerank<CL>(c, L, crank, &rr_cycles)) return;
  Pwl P;
  make_pwl(P, L.prm[c.s]);
  improve(c, L, P);
  double me_all = 0.0;
  const long long shortf_all = objective(c, L, P, rr_cycles, &me_all);
  if (L.ncap && shortf_all > 0) packing_feedback(c, L, P, me_all, shortf_all);
  backfill(c, L);
  __syncthreads();
  write_outputs(c, L);
}

// The whole launch decision of one call's placement.
PlacePlan plan_place(int S, int J, int T, int rr_iters, int cluster_opt) {
  PlacePlan pl = {};
  PlaceSmem m;
  RrScratch r;
  pl.rr_region = rr_carve(r, nullptr, nullptr, J, T);
  // re-rank local search: O(J T^2) per cancelled cycle — on where that stays in the tens of microseconds (jobs x
  // rounds^2 <= 256 Ki: 640 jobs at 20 rounds, 250 at 32, 64 at 64 — the reference's deployments; beyond that the
  // priority sweep alone places the fallback schedule), and with the round masks in shared memory
  pl.rerank = rr_iters > 0 && J <= SWB_SMEM_JOBS && (size_t)J * T * T <= (256u << 10);
  // multi-start over a cluster of 8 CTAs per scenario while the launch still fits one wave of SMs
  pl.cluster = (pl.rerank && cluster_opt == 8 && S * 8 <= 144) ? 8 : 1;
  pl.rr_bytes = pl.rerank ? (size_t)S * pl.cluster * pl.rr_region : 0;
  if (pl.rr_bytes > (512u << 20)) { pl.rerank = 0; pl.cluster = 1; pl.rr_bytes = 0; }
  const int npad = sort_pad(J);
  pl.threads = npad < SWB_PLACE_THREADS ? npad : SWB_PLACE_THREADS;
  pl.smem = place_carve(m, nullptr, J, T, false);
  if (pl.rerank) {
    // the search wants a thread per ordered pair of rounds; its hot arrays go to shared memory when they fit (up to
    // about 80 rounds), else the search reads them from its scratch
    if (pl.threads < 512) pl.threads = 512;
    const size_t hot = place_carve(m, nullptr, J, T, true);
    int stat = 0;
    { cudaFuncAttributes fa; if (cudaFuncGetAttributes(&fa, place_kernel<1>) == cudaSuccess) stat = (int)fa.sharedSizeBytes; }
    if (hot + (size_t)stat <= (size_t)SWB_MAX_DYN_SMEM) { pl.smem = hot; pl.hot_smem = 1; }
  }
  return pl;
}

cudaError_t launch_place(const PlaceLaunch &L, cudaStream_t st, unsigned long long *gmask) {
  // function attributes are per device: one flag per device ordinal (one process may drive several GPUs)
  static bool attr_done[64] = {false};
  int dev_ = 0;
  cudaGetDevice(&dev_);
  bool &attr_set = attr_done[dev_ & 63];
  if (!attr_set) {
    cudaFuncAttributes fa;
    cudaError_t e = cudaFuncGetAttributes(&fa, place_kernel<1>);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(place_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             SWB_MAX_DYN_SMEM - (int)fa.sharedSizeBytes);
    if (e != cudaSuccess) return e;
    e = cudaFuncGetAttributes(&fa, place_kernel<8>);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(place_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             SWB_MAX_DYN_SMEM - (int)fa.sharedSizeBytes);
    if (e != cudaSuccess) return e;
    attr_set = true;
  }
  const PlacePlan &pl = L.plan;
  if (pl.cluster == 8) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(L.S * 8)); cfg.blockDim = dim3((unsigned)pl.threads);
    cfg.dynamicSmemBytes = pl.smem; cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = 8; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, place_kernel<8>, L, gmask);
  }
  place_kernel<1><<<L.S, pl.threads, pl.smem, st>>>(L, gmask);
  return cudaGetLastError();
}

}  // namespace swb
