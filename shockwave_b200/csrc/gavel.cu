// gavel.cu — Gavel's per-round priority -> selection -> worker-assignment step on one B200 (sm_100a), one launch.
//
// Reference behaviour replaced (the step right after policy.get_allocation(), SURVEY.md §8(f)-2):
//   priorities   scheduler/scheduler.py:3669-3724  fraction of worker time received vs. allocation
//   selection    scheduler/scheduler.py:1166-1258  per worker type: stable sort by (priority, deficit, allocation)
//                                                   descending, then a greedy walk that skips what does not fit
//   assignment   scheduler/scheduler.py:1306-1378, :1049-1110  largest scale factor first; a job keeps last round's
//                                                   workers when they are all still free (lease extension), the rest
//                                                   take the next free workers in server order
// All of it is integer / comparison work on per-(job, type) float64 scalars: the priorities use the reference's own
// IEEE operations (one division), the sort is a bitonic network over job indices with the reference's lexicographic
// key and the original index as the last key (= Python's stable sort), the greedy walk is resolved in a few parallel
// passes (jobs wider than what is left can never fit later; of the rest the longest prefix that fits is taken at
// once), and worker assignment is two prefix scans per scale-factor class.  Results are bit-for-bit those of the dict
// code (tests/test_gpu_gavel_round.py against oracle/gavel_round.py, itself pinned on the golden pickles).
// One CTA; J <= 8192 jobs, W <= 8 worker types, <= 8192 workers per type.
#include <math.h>

#include "swb_common.cuh"
#include "swb_internal.h"

namespace swb {

// a before b in the reference's queue: (priority, deficit, allocation) descending, ties in dict order
__device__ __forceinline__ bool gv_before(const GavelLaunch &L, int w, int a, int b) {
  if (a >= L.J || b >= L.J) return a < b;          // padding sorts last
  const size_t ia = (size_t)a * L.W + w, ib = (size_t)b * L.W + w;
  const double pa = L.prio[ia], pb = L.prio[ib];
  if (pa != pb) return pa > pb;
  const double da = L.deficit[ia], db = L.deficit[ib];
  if (da != db) return da > db;
  double xa = L.alloc[ia], xb = L.alloc[ib];
  xa = isnan(xa) ? 0.0 : xa; xb = isnan(xb) ? 0.0 : xb;     // job not in the allocation: 0.0 (scheduler.py:1177-1183)
  if (xa != xb) return xa > xb;
  return a < b;
}

__global__ void __launch_bounds__(1024, 1) gavel_round_kernel(GavelLaunch L) {
  extern __shared__ __align__(16) unsigned char smem[];
  const int J = L.J, W = L.W, tid = threadIdx.x, nt = blockDim.x;
  int npad = 64;
  while (npad < J) npad <<= 1;
  unsigned short *ord = reinterpret_cast<unsigned short *>(smem);            // [npad] sorted job indices
  unsigned char *state = smem + 2 * (size_t)npad;                            // [npad] per job (see below)
  unsigned char *wbusy = state + npad;                                       // [maxw] worker of this type assigned
  int *wsum = reinterpret_cast<int *>((reinterpret_cast<uintptr_t>(wbusy + L.maxw) + 15) & ~uintptr_t(15));
  __shared__ int s_left, s_stop, s_nsel, s_nasg, s_err;
  __shared__ double s_red[2 * 64];
  BlockRed br(s_red);
  // per-job flags, global scratch: bit0 = scheduled on some type already
  unsigned char *sched = L.sched;

  // ---- 1. priorities (scheduler.py:3669-3724) ---------------------------------------------------------------
  for (int e = tid; e < J * W; e += nt) {
    const int w = e % W;
    const double a = L.alloc[e];
    double p = 0.0;
    if (!isnan(a)) {
      const double wt = L.worker_time[w];
      const double fraction = (wt == 0.0) ? 0.0 : L.job_time[e] / wt;
      p = a * 1e9;
      if (a == 0.0) p = 0.0;
      else if (L.thr[e] == 0.0) p = 0.0;
      else if (fraction > 0.0) p = a / fraction;
    }
    L.prio[e] = p;
  }
  // sched[j]: bit 0 = scheduled on some type already, bit 1 = the allocation knows the job (any non-NaN entry)
  for (int j = tid; j < J; j += nt) {
    unsigned char known = 0;
    for (int w = 0; w < W; ++w) known |= isnan(L.alloc[(size_t)j * W + w]) ? 0 : 2;
    sched[j] = known;
  }
  if (tid == 0) { s_stop = 0; s_nasg = 0; s_err = 0; L.assign_off[0] = 0; }
  __syncthreads();

  int woff_type = 0;     // offset of this type's workers in worker_ids (types are stored in processing order)
  for (int ti = 0; ti < W; ++ti) {
    const int w = L.type_order[ti];
    const int nw = L.nworkers[ti];
    // ---- 2. the type's queue: stable sort by (priority, deficit, allocation) descending ---------------------
    if (s_stop) { if (tid == 0) L.n_sel[ti] = 0; woff_type += nw; continue; }   // Isolated_plus: the walk has ended
    for (int i = tid; i < npad; i += nt) ord[i] = (unsigned short)i;
    __syncthreads();
    for (int k = 2; k <= npad; k <<= 1)
      for (int jj = k >> 1; jj > 0; jj >>= 1) {
        for (int i = tid; i < npad; i += nt) {
          const int p = i ^ jj;
          if (p > i) {
            const int a = ord[i], b = ord[p];
            const bool a_first = gv_before(L, w, a, b);
            const bool up = (i & k) == 0;
            if (up != a_first) { ord[i] = (unsigned short)b; ord[p] = (unsigned short)a; }
          }
        }
        __syncthreads();
      }
    // ---- 3. greedy walk (scheduler.py:1212-1258).  state[pos]: 0 = candidate, 1 = taken, 2 = rejected ---------
    if (tid == 0) { s_left = L.capacity[w]; s_nsel = 0; }
    const int chs = (npad + nt - 1) / nt, p0 = tid * chs;
    for (int q = 0; q < chs; ++q) {
      const int pos = p0 + q;
      if (pos < npad) {
        const int j = ord[pos];
        unsigned char st = 2;
        if (j < J && !(sched[j] & 1) && L.thr[(size_t)j * W + w] > 0.0 &&
            !((L.flags & 2) && L.prio[(size_t)j * W + w] <= 0.0))
          st = 0;
        state[pos] = st;
      }
    }
    __syncthreads();
    if (L.flags & 1) {
      // Isolated_plus: strict priority order — the walk (over ALL worker types) ends at the first candidate that does
      // not fit (scheduler.py:1243-1250); a running sum over the candidates finds it in one pass
      int lsum = 0;
      for (int q = 0; q < chs; ++q) { const int pos = p0 + q; if (pos < npad && state[pos] == 0) lsum += L.sf[ord[pos]]; }
      int tot = 0;
      int run = block_excl_scan(lsum, wsum, &tot);
      const int left = s_left;
      int stop = 0;
      for (int q = 0; q < chs; ++q) {
        const int pos = p0 + q;
        if (pos < npad && state[pos] == 0) {
          const int s = L.sf[ord[pos]];
          run += s;
          if (run <= left) state[pos] = 1;
          else if (run - s < left) stop = 1;     // workers were left at its turn and it did not fit: `break`
        }                                        // (with none left the reference only `continue`s, :1213-1214)
      }
      stop = __syncthreads_or(stop);
      if (tid == 0 && stop) s_stop = 1;
      __syncthreads();
    } else {
      for (int pass = 0; pass < 4096; ++pass) {
        const int left = s_left;
        if (left == 0) break;
        // candidates wider than what is left can never fit later (left only shrinks): rejected for good
        int lsum = 0;
        for (int q = 0; q < chs; ++q) {
          const int pos = p0 + q;
          if (pos < npad && state[pos] == 0) {
            const int s = L.sf[ord[pos]];
            if (s > left) state[pos] = 2; else lsum += s;
          }
        }
        int tot = 0;
        int run = block_excl_scan(lsum, wsum, &tot);
        if (tot == 0) break;
        // the longest prefix that fits is taken at once; the first candidate beyond it does not fit what is then left
        // and is rejected by the width test of the next pass
        int took = 0;
        for (int q = 0; q < chs; ++q) {
          const int pos = p0 + q;
          if (pos < npad && state[pos] == 0) {
            const int s = L.sf[ord[pos]];
            run += s;
            if (run <= left) { state[pos] = 1; took += s; }
          }
        }
        const int taken = br.sumi(took);
        if (tid == 0) s_left = left - taken;
        __syncthreads();
        if (taken == tot) break;
      }
    }
    __syncthreads();
    // selection order = queue order of the taken positions
    {
      int cnt = 0;
      for (int q = 0; q < chs; ++q) { const int pos = p0 + q; if (pos < npad && state[pos] == 1) ++cnt; }
      int tot = 0;
      int off = block_excl_scan(cnt, wsum, &tot);
      for (int q = 0; q < chs; ++q) {
        const int pos = p0 + q;
        if (pos < npad && state[pos] == 1) { const int j = ord[pos]; L.sel_jobs[(size_t)ti * J + off++] = j; sched[j] |= 1; }
      }
      if (tid == 0) { s_nsel = tot; L.n_sel[ti] = tot; }
    }
    __syncthreads();
    // ---- 4. worker assignment, largest scale factor first (scheduler.py:1306-1378) ------------------------------
    const int nsel = s_nsel;
    const int32_t *sel = L.sel_jobs + (size_t)ti * J;
    const int32_t *wids = L.worker_ids + woff_type;
    for (int i = tid; i < nw; i += nt) wbusy[i] = 0;
    // state[i] for i < nsel: 0 = pending, 1 = done (reused: positions now index the selection list)
    for (int i = tid; i < nsel; i += nt) state[i] = 0;
    __syncthreads();
    int cur = 1 << 30;
    for (int cls = 0; cls < 64; ++cls) {
      // next class: the largest scale factor below `cur`
      int m = 0;
      for (int i = tid; i < nsel; i += nt) { const int s = L.sf[sel[i]]; if (s < cur && s > m) m = s; }
      m = (int)br.max((double)m);
      if (m <= 0) break;
      cur = m;
      // (a) lease extension: previous workers of this type, all still free (previous assignments are disjoint, so
      //     jobs of one class cannot collide with each other)
      const int chn = (nsel + nt - 1) / nt, n0 = tid * chn;
      int cntA = 0;
      for (int q = 0; q < chn; ++q) {
        const int i = n0 + q;
        if (i < nsel) {
          const int j = sel[i];
          if (L.sf[j] == cur && L.prev_type[j] == w) {
            bool ok = true;
            for (int e = L.prev_off[j]; e < L.prev_off[j + 1]; ++e) {
              const int lw = L.prev_local[e];
              if (lw < 0 || lw >= nw || wbusy[lw]) { ok = false; break; }
            }
            if (ok) { state[i] = 2; ++cntA; }
          }
        }
      }
      __syncthreads();
      int totA = 0;
      int offA = block_excl_scan(cntA, wsum, &totA);
      const int baseA = s_nasg;
      for (int q = 0; q < chn; ++q) {
        const int i = n0 + q;
        if (i < nsel && state[i] == 2) {
          const int j = sel[i];
          const int slot = baseA + offA++;
          L.assign_job[slot] = j;
          L.assign_cnt[slot] = L.prev_off[j + 1] - L.prev_off[j];
          for (int e = L.prev_off[j]; e < L.prev_off[j + 1]; ++e) wbusy[L.prev_local[e]] = 1;
          state[i] = 3;     // extended; workers written below once the offsets are known
        }
      }
      __syncthreads();
      // (b) the class's remaining jobs (only those the allocation knows, scheduler.py:1364-1368) take the next free
      //     workers in server order
      int cntB = 0, needB = 0;
      for (int q = 0; q < chn; ++q) {
        const int i = n0 + q;
        if (i < nsel && state[i] == 0 && L.sf[sel[i]] == cur && (sched[sel[i]] & 2)) { ++cntB; needB += cur; }
      }
      int totB = 0, totNeed = 0;
      int offB = block_excl_scan(cntB, wsum, &totB);
      int offNeed = block_excl_scan(needB, wsum, &totNeed);
      // free workers in order: rank of every free worker
      const int chw = (nw + nt - 1) / nt, w0 = tid * chw;
      int cntF = 0;
      for (int q = 0; q < chw; ++q) { const int i = w0 + q; if (i < nw && !wbusy[i]) ++cntF; }
      int totF = 0;
      int offF = block_excl_scan(cntF, wsum, &totF);
      if (totNeed > totF) { if (tid == 0) s_err = 1; __syncthreads(); break; }
      const int baseB = baseA + totA;
      // every free worker with rank < totNeed goes to the job whose [offNeed, offNeed + cur) range covers the rank:
      // rank / cur-th pending job of the class (all have the same width)
      for (int q = 0; q < chn; ++q) {
        const int i = n0 + q;
        if (i < nsel && state[i] == 0 && L.sf[sel[i]] == cur && (sched[sel[i]] & 2)) {
          const int slot = baseB + offB++;
          L.assign_job[slot] = sel[i];
          L.assign_cnt[slot] = cur;
          L.tmp_rank0[slot] = offNeed; offNeed += cur;
          state[i] = 4;
        }
      }
      __syncthreads();
      // scatter: free worker of rank r -> slot baseB + r / cur, position r % cur
      for (int q = 0; q < chw; ++q) {
        const int i = w0 + q;
        if (i < nw && !wbusy[i]) {
          const int r = offF++;
          if (r < totNeed) L.tmp_free[r] = i;
        }
      }
      __syncthreads();
      for (int r = tid; r < totNeed; r += nt) wbusy[L.tmp_free[r]] = 1;
      // mark skipped jobs (not in the allocation) done
      for (int q = 0; q < chn; ++q) {
        const int i = n0 + q;
        if (i < nsel && state[i] == 0 && L.sf[sel[i]] == cur) state[i] = 5;
      }
      __syncthreads();
      // offsets + worker ids of the class's assignments, in insertion order (extended first, then the rest)
      if (tid == 0) {
        int o = L.assign_off[baseA];
        for (int sl = baseA; sl < baseB + totB; ++sl) { o += L.assign_cnt[sl]; L.assign_off[sl + 1] = o; }
        s_nasg = baseB + totB;
      }
      __syncthreads();
      for (int sl = baseA + tid; sl < baseB + totB; sl += nt) {
        const int j = L.assign_job[sl], o = L.assign_off[sl];
        if (sl < baseB) {
          int k = 0;
          for (int e = L.prev_off[j]; e < L.prev_off[j + 1]; ++e) L.assign_workers[o + k++] = wids[L.prev_local[e]];
        } else {
          const int r0 = L.tmp_rank0[sl];
          for (int k = 0; k < cur; ++k) L.assign_workers[o + k] = wids[L.tmp_free[r0 + k]];
        }
      }
      __syncthreads();
    }
    if (s_err) break;
    woff_type += nw;
    __syncthreads();
  }
  if (tid == 0) { L.out_scalars[0] = s_nasg; L.out_scalars[1] = s_err; }
}

cudaError_t launch_gavel_round(const GavelLaunch &L, cudaStream_t st) {
  int npad = 64;
  while (npad < L.J) npad <<= 1;
  const size_t smem = 2 * (size_t)npad + npad + (size_t)L.maxw + 16 + 64 * sizeof(int) + 64;
  static bool attr_done[64] = {false};
  int dev_ = 0;
  cudaGetDevice(&dev_);
  if (!attr_done[dev_ & 63]) {
    cudaError_t e = cudaFuncSetAttribute(gavel_round_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    if (e != cudaSuccess) return e;
    attr_done[dev_ & 63] = true;
  }
  int nt = npad < 1024 ? npad : 1024;
  gavel_round_kernel<<<1, nt, smem, st>>>(L);
  return cudaGetLastError();
}

}  // namespace swb
