"""ctypes binding of libswb200.so (the C-ABI declared in include/swb200.h).

This is the only place the product touches the shared library.  There is NO CPU path: if the
library is missing or no B200 is visible, constructing an `Engine` raises.  numpy arrays are the
host containers; raw device pointers (e.g. `torch.Tensor.data_ptr()`) are accepted where the header
says `on_device`.
"""
from __future__ import annotations

import ctypes as C
import math
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libswb200.so")

MAX_BASES = 16
ST_OK, ST_FALLBACK = 0, 1
OPT_RELAXED_OPTIMUM, OPT_SOLVE_CLUSTER, OPT_GBM_PATHS, OPT_GBM_SEED, OPT_GBM_HORIZON, OPT_RERANK_ITERS, OPT_RERANK_RESTARTS, OPT_ASYNC_AUX = 1, 2, 3, 4, 5, 6, 7, 8


class Params(C.Structure):
    """swb_params (include/swb200.h)."""
    _fields_ = [("ngpus", C.c_int32), ("future_rounds", C.c_int32), ("round_ptr", C.c_int32),
                ("nbases", C.c_int32), ("round_duration", C.c_double), ("k", C.c_double),
                ("lam", C.c_double), ("rhomax", C.c_double),
                ("bases", C.c_double * MAX_BASES), ("logv", C.c_double * MAX_BASES)]


class Result(C.Structure):
    """swb_result (include/swb200.h)."""
    _fields_ = [("status", C.c_int32), ("m_evals", C.c_int32), ("mu_iters", C.c_int32),
                ("shortfall", C.c_int32), ("placement", C.c_int32), ("flags", C.c_int32),
                ("objective", C.c_double), ("welfare", C.c_double),
                ("makespan", C.c_double), ("price", C.c_double), ("relaxed_objective", C.c_double)]

    def as_dict(self):
        return {f: getattr(self, f) for f, _ in self._fields_}


class SolveArgs(C.Structure):
    """swb_solve_args (include/swb200.h)."""
    _fields_ = [("S", C.c_int32), ("J", C.c_int32), ("per_scenario_jobs", C.c_int32),
                ("on_device", C.c_int32), ("prm", C.POINTER(Params)),
                ("g", C.c_void_p), ("E", C.c_void_p), ("c", C.c_void_p),
                ("dbar", C.c_void_p), ("rem", C.c_void_p), ("ftobj", C.c_void_p), ("bfkey", C.c_void_p),
                ("x", C.c_void_p), ("backfill", C.c_void_p), ("nrounds", C.c_void_p),
                ("weights", C.c_void_p), ("res", C.POINTER(Result)), ("xmask", C.c_void_p), ("bfmask", C.c_void_p)]


class RoundArgs(C.Structure):
    """swb_round_args (include/swb200.h)."""
    _fields_ = [("J", C.c_int32), ("reestimate_share", C.c_int32), ("gavel_round_duration", C.c_double),
                ("slots", C.c_void_p), ("epoch_progress", C.c_void_p), ("meas_nsamples", C.c_void_p),
                ("meas_end_round", C.c_void_p), ("x", C.c_void_p), ("backfill", C.c_void_p),
                ("nrounds", C.c_void_p), ("forecast_out", C.c_void_p), ("res", C.POINTER(Result)),
                ("xmask", C.c_void_p), ("bfmask", C.c_void_p)]


class MarketArgs(C.Structure):
    """swb_market_args (include/swb200.h)."""
    _fields_ = [("S", C.c_int32), ("J", C.c_int32), ("W", C.c_int32), ("T", C.c_int32),
                ("per_scenario_jobs", C.c_int32), ("on_device", C.c_int32), ("iters", C.c_int32),
                ("coarse_iters", C.c_int32), ("warm_start", C.c_int32), ("primal_weight", C.c_float), ("utility", C.c_int32),
                ("prm", C.POINTER(Params)), ("g", C.c_void_p), ("E", C.c_void_p), ("c", C.c_void_p),
                ("dbar", C.c_void_p), ("rem", C.c_void_p), ("rate", C.c_void_p), ("Gw", C.c_void_p),
                ("cap", C.c_void_p), ("X", C.c_void_p), ("obj", C.c_void_p), ("dense_ms", C.POINTER(C.c_float))]


class GavelRoundArgs(C.Structure):
    """swb_gavel_round_args (include/swb200.h)."""
    _fields_ = [("J", C.c_int32), ("W", C.c_int32), ("flags", C.c_int32)] + \
               [(n, C.c_void_p) for n in ("type_order", "capacity", "alloc", "job_time", "thr", "deficit",
                                          "worker_time", "sf", "nworkers", "worker_ids", "prev_type", "prev_off",
                                          "prev_local", "prio", "n_sel", "sel_jobs")] + \
               [("n_assigned", C.POINTER(C.c_int32))] + \
               [(n, C.c_void_p) for n in ("assign_job", "assign_off", "assign_workers")]


class SimTrace(C.Structure):
    """swb_sim_trace (include/swb200.h)."""
    _fields_ = [("J", C.c_int32), ("reserved", C.c_int32), ("arrival", C.c_void_p), ("total_steps", C.c_void_p),
                ("scale_factor", C.c_void_p), ("throughput", C.c_void_p), ("duration", C.c_void_p),
                ("batch_size", C.c_void_p), ("dataset_len", C.c_void_p), ("adaptation_mode", C.c_void_p)]


class SimDynamic(C.Structure):
    """swb_sim_dynamic (include/swb200.h)."""
    _fields_ = [("mode", C.c_void_p), ("bs_max", C.c_void_p), ("bs_min", C.c_void_p), ("bs_big", C.c_void_p),
                ("orig_locked", C.c_void_p), ("acc_skip", C.c_void_p), ("pat_off", C.c_void_p), ("pattern", C.c_void_p),
                ("n_levels", C.c_int32), ("reserved", C.c_int32), ("lvl_bs", C.c_void_p), ("lvl_thr", C.c_void_p)]


class SimScn(C.Structure):
    """swb_sim_scn (include/swb200.h)."""
    _fields_ = [("now", C.c_double), ("round_start", C.c_double), ("round_end", C.c_double), ("rounds", C.c_int32),
                ("remaining", C.c_int32), ("n_active", C.c_int32), ("done", C.c_int32), ("err", C.c_int32),
                ("reserved", C.c_int32)]


SCN_DTYPE = np.dtype([("now", "f8"), ("round_start", "f8"), ("round_end", "f8"), ("rounds", "i4"), ("remaining", "i4"),
                      ("n_active", "i4"), ("done", "i4"), ("err", "i4"), ("reserved", "i4")])   # numpy view of SimScn
assert SCN_DTYPE.itemsize == C.sizeof(SimScn) == 48

# Every function include/swb200.h declares: name -> (restype, argtypes).  load_library() binds the whole table;
# tests/test_abi_and_host.py checks it against the header's prototypes.
_P, _I32, _I64, _F64, _PF64 = C.c_void_p, C.c_int32, C.c_int64, C.c_double, C.POINTER(C.c_double)
ABI = {
    "swb_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_int]),
    "swb_destroy": (None, [_P]),
    "swb_last_error": (C.c_char_p, []),
    "swb_version": (C.c_int, []),
    "swb_stream": (C.c_void_p, [_P]),
    "swb_sync": (C.c_int, [_P]),
    "swb_set_option": (C.c_int, [_P, _I32, _I32]),
    "swb_solve": (C.c_int, [_P, C.POINTER(SolveArgs)]),
    "swb_job_add": (C.c_int, [_P, _I32, _I32, _I32, _F64, _F64, _P, _P]),
    "swb_job_remove": (C.c_int, [_P, _I32]),
    "swb_job_table_stats": (C.c_int, [_P, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "swb_job_set_gbm": (C.c_int, [_P, _I32, _F64, _F64]),
    "swb_round_solve": (C.c_int, [_P, C.POINTER(Params), C.POINTER(RoundArgs)]),
    "swb_forecast": (C.c_int, [_P, C.POINTER(Params), C.POINTER(RoundArgs)] + [_P] * 5),
    "swb_forecast_commit": (C.c_int, [_P, _I32, _I32, _P]),
    "swb_policy_pooled": (C.c_int, [_P, _I32, _I32, _F64] + [_P] * 6 + [_PF64]),
    "swb_policy_hetero": (C.c_int, [_P, _I32, _I32, _I32] + [_P] * 7 + [_PF64, _P]),
    "swb_policy_waterfill_step": (C.c_int, [_P, _I32, _I32] + [_P] * 6 + [_F64, _F64, _P, _PF64, _P, _P]),
    "swb_lp_solve": (C.c_int, [_P] + [_I32] * 4 + [_P] * 5 + [_I32] + [_P] * 4),
    "swb_allox_assign": (C.c_int, [_P, _I32, _I32, _I32] + [_P] * 4 + [_PF64]),
    "swb_gavel_round": (C.c_int, [_P, C.POINTER(GavelRoundArgs)]),
    "swb_gbm_forecast": (C.c_int, [_P, _I32] + [_P] * 4 + [_I64, _I64, C.c_uint64, _P, _I32]),
    "swb_gbm_ensemble": (C.c_int, [_P, _I32, _I32, _F64, _P, _P, _P]),
    "swb_market_pgd": (C.c_int, [_P, C.POINTER(MarketArgs)]),
    "swb_sim_set_dynamic": (C.c_int, [_P, C.POINTER(SimDynamic)]),
    "swb_sim_set_worker_types": (C.c_int, [_P, _I32, _P, _P]),
    "swb_sim_create": (C.c_int, [_I32, C.POINTER(SimTrace), _I32, _I32, _F64, _F64, C.POINTER(C.c_void_p)]),
    "swb_sim_destroy": (None, [_P]),
    "swb_sim_begin": (C.c_int, [_P, _P, _P]),
    "swb_sim_step": (C.c_int, [_P] * 7),
    "swb_sim_replay": (C.c_int, [_P, _P, _I32, _I32, _P]),
    "swb_sim_results": (C.c_int, [_P] * 5),
    "swb_sim_job_state": (C.c_int, [_P] * 8),
    "swb_last_timings": (C.c_int, [_P, _PF64, _PF64, C.POINTER(C.c_int32)]),
}
EXPORTS = list(ABI)

_lib = None


def load_library():
    """dlopen libswb200.so; raises (never falls back) when it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(there is no CPU fallback for the shockwave_b200 solver)")
    lib = C.CDLL(LIB_PATH)
    for name, (restype, argtypes) in ABI.items():
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = restype, argtypes
    _lib = lib
    return lib


def make_params(ngpus, future_rounds, round_duration, k, lam, rhomax, bases, origin, round_ptr=0):
    """swb_params from the ShockwaveScheduler constructor kwargs (shockwave.py:21-86)."""
    p = Params()
    p.ngpus, p.future_rounds, p.round_ptr, p.nbases = int(ngpus), int(future_rounds), int(round_ptr), len(bases)
    p.round_duration, p.k, p.lam, p.rhomax = float(round_duration), float(k), float(lam), float(rhomax)
    assert bases[0] == 0.0 and len(bases) <= MAX_BASES
    for i, b in enumerate(bases):
        assert 0.0 <= b <= 1.0
        p.bases[i] = float(b)
        p.logv[i] = math.log(origin[0.0]) if b == 0.0 else math.log(b)   # shockwave.py:339-347
    return p


def _ptr(a):
    return None if a is None else C.c_void_p(a.ctypes.data)


def unpack_masks(mask, T):
    """[..., J, 2] uint64 round masks -> [..., J, T] uint8 (bit t of the 128-bit row = round t)."""
    b = np.unpackbits(np.ascontiguousarray(mask).view(np.uint8), axis=-1, bitorder="little")
    return b.reshape(mask.shape[:-1] + (128,))[..., :T]


class Engine:
    """One swb_ctx (one CUDA stream on one B200)."""

    def __init__(self, device=0):
        self.lib = load_library()
        h = C.c_void_p()
        rc = self.lib.swb_create(C.byref(h), int(device))
        if rc != 0:
            raise RuntimeError(f"swb_create failed ({rc}): {self.lib.swb_last_error().decode()}")
        self.h = h

    def close(self):
        if getattr(self, "h", None):
            self.lib.swb_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, what):
        if rc < 0:
            raise RuntimeError(f"{what} failed ({rc}): {self.lib.swb_last_error().decode()}")
        return rc

    # ---- plain-array market solve (swb_solve) -----------------------------------------------------
    def solve(self, params, g, E, c, dbar, rem, ftobj, bfkey=None, want_x=True, want_backfill=True, packed=False,
              out=None):
        """Solve S scenarios on host arrays.  `params`: one Params or a list of S; per-job arrays are
        [J] (shared) or [S, J].  Returns dict(x[S,J,T] u8, backfill, nrounds, weights, results[list])."""
        plist = params if isinstance(params, (list, tuple)) else [params]
        S = len(plist)
        g = np.ascontiguousarray(g, dtype=np.int32)
        per = 1 if g.ndim == 2 else 0
        J = g.shape[-1]
        E = np.ascontiguousarray(E, dtype=np.int32); c = np.ascontiguousarray(c, dtype=np.int32)
        dbar = np.ascontiguousarray(dbar, dtype=np.float64); rem = np.ascontiguousarray(rem, dtype=np.float64)
        ftobj = np.ascontiguousarray(ftobj, dtype=np.float64)
        bfkey = rem if bfkey is None else np.ascontiguousarray(bfkey, dtype=np.float64)
        for a in (E, c, dbar, rem, ftobj, bfkey):
            assert a.shape == g.shape
        T = plist[0].future_rounds
        parr = (Params * S)(*plist)
        res = (Result * S)()
        # packed=True: 128-bit round masks instead of the byte matrices (16 B/job instead of T B/job on the
        # device->host copy); unpack with unpack_masks().  `out`: preallocated (e.g. pinned) output arrays.
        out = out or {}
        x = bf = xm = bm = None
        if packed:
            xm = out.get("xmask") if out.get("xmask") is not None else np.zeros((S, J, 2), dtype=np.uint64)
            bm = out.get("bfmask") if out.get("bfmask") is not None else np.zeros((S, J, 2), dtype=np.uint64)
        else:
            x = np.zeros((S, J, T), dtype=np.uint8) if want_x else None
            bf = np.zeros((S, J, T), dtype=np.uint8) if want_backfill else None
        nr = out.get("nrounds") if out.get("nrounds") is not None else np.zeros((S, J), dtype=np.int32)
        w = out.get("weights") if out.get("weights") is not None else np.zeros((S, J), dtype=np.float64)
        a = SolveArgs(S, J, per, 0, parr, _ptr(g), _ptr(E), _ptr(c), _ptr(dbar), _ptr(rem), _ptr(ftobj),
                      _ptr(bfkey), _ptr(x), _ptr(bf), _ptr(nr), _ptr(w), res, _ptr(xm), _ptr(bm))
        self._check(self.lib.swb_solve(self.h, C.byref(a)), "swb_solve")
        return dict(x=x, backfill=bf, xmask=xm, bfmask=bm, nrounds=nr, weights=w,
                    results=[r.as_dict() for r in res])

    def solve_device(self, params, J, ptrs, out_ptrs, per_scenario_jobs=True):
        """Same on raw DEVICE pointers (ints): ptrs = dict(g,E,c,dbar,rem,ftobj,bfkey),
        out_ptrs = dict(x, backfill, nrounds, weights) (0/None = not wanted)."""
        plist = params if isinstance(params, (list, tuple)) else [params]
        S = len(plist)
        parr = (Params * S)(*plist)
        res = (Result * S)()
        vp = lambda v: C.c_void_p(int(v)) if v else None
        a = SolveArgs(S, J, 1 if per_scenario_jobs else 0, 1, parr, vp(ptrs["g"]), vp(ptrs["E"]), vp(ptrs["c"]),
                      vp(ptrs["dbar"]), vp(ptrs["rem"]), vp(ptrs["ftobj"]), vp(ptrs.get("bfkey")),
                      vp(out_ptrs.get("x")), vp(out_ptrs.get("backfill")), vp(out_ptrs.get("nrounds")),
                      vp(out_ptrs.get("weights")), res, vp(out_ptrs.get("xmask")), vp(out_ptrs.get("bfmask")))
        self._check(self.lib.swb_solve(self.h, C.byref(a)), "swb_solve")
        return [r.as_dict() for r in res]

    # ---- resident job table -------------------------------------------------------------------------
    def job_add(self, slot, nworkers, epochs, epoch_nsamples, timestamp_submit, epoch_duration_pre, bs_schedule):
        pre = np.ascontiguousarray(epoch_duration_pre, dtype=np.float64)
        bs = np.ascontiguousarray(bs_schedule, dtype=np.int32)
        assert len(pre) == len(bs) == int(epochs)
        self._check(self.lib.swb_job_add(self.h, int(slot), int(nworkers), int(epochs), float(epoch_nsamples),
                                         float(timestamp_submit), _ptr(pre), _ptr(bs)), "swb_job_add")

    def job_remove(self, slot):
        self._check(self.lib.swb_job_remove(self.h, int(slot)), "swb_job_remove")

    def job_set_gbm(self, slot, mu, sigma):
        self._check(self.lib.swb_job_set_gbm(self.h, int(slot), float(mu), float(sigma)), "swb_job_set_gbm")

    def gbm_ensemble(self, S, J, P_total, sums_device_ptr, z, rem_out_device_ptr):
        z = np.ascontiguousarray(z, dtype=np.float64)
        assert len(z) == S
        self._check(self.lib.swb_gbm_ensemble(self.h, int(S), int(J), float(P_total), C.c_void_p(int(sums_device_ptr)),
                                              _ptr(z), C.c_void_p(int(rem_out_device_ptr))), "swb_gbm_ensemble")

    def gavel_round(self, alloc, job_time, worker_time, thr, deficit, sf, capacity, type_order, worker_lists, prev,
                    isolated_plus=False, fifo=False):
        """swb_gavel_round on plain arrays.  alloc / job_time / thr / deficit: [J, W] float64 (alloc NaN = job not in
        the allocation); worker_lists: list (processing order) of flat worker-id lists; prev: {job idx: (type idx,
        (worker ids))}.  Returns (prio [J, W], {type idx: [job idx in selection order]}, [(job idx, (worker ids))] in
        the reference's insertion order)."""
        f64 = lambda v: np.ascontiguousarray(v, dtype=np.float64)
        i32 = lambda v: np.ascontiguousarray(v, dtype=np.int32)
        alloc, job_time, thr, deficit, worker_time = f64(alloc), f64(job_time), f64(thr), f64(deficit), f64(worker_time)
        J, W = alloc.shape
        sf, capacity, type_order = i32(sf), i32(capacity), i32(type_order)
        nworkers = i32([len(wl) for wl in worker_lists])
        wids = i32([w for wl in worker_lists for w in wl]) if nworkers.sum() else np.zeros(1, np.int32)
        local = [{w: i for i, w in enumerate(worker_lists[ti])} for ti in range(W)]
        pos_of_type = {int(t): ti for ti, t in enumerate(type_order)}
        prev_type = np.full(J, -1, dtype=np.int32)
        prev_off = np.zeros(J + 1, dtype=np.int32)
        pl = []
        for j in range(J):
            if j in prev:
                t, ws = prev[j]
                prev_type[j] = t
                lut = local[pos_of_type[int(t)]] if int(t) in pos_of_type else {}
                pl += [lut.get(w, -1) for w in ws]
            prev_off[j + 1] = len(pl)
        prev_local = i32(pl) if pl else np.zeros(1, np.int32)
        prio = np.empty((J, W), dtype=np.float64)
        n_sel = np.zeros(W, dtype=np.int32); sel_jobs = np.zeros((W, J), dtype=np.int32)
        n_asg = C.c_int32(); a_job = np.zeros(J, dtype=np.int32); a_off = np.zeros(J + 1, dtype=np.int32)
        a_w = np.zeros(max(1, int(nworkers.sum())), dtype=np.int32)
        a = GavelRoundArgs(J, W, (1 if isolated_plus else 0) | (2 if fifo else 0), _ptr(type_order), _ptr(capacity), _ptr(alloc),
                 _ptr(job_time), _ptr(thr), _ptr(deficit), _ptr(worker_time), _ptr(sf), _ptr(nworkers), _ptr(wids),
                 _ptr(prev_type), _ptr(prev_off), _ptr(prev_local), _ptr(prio), _ptr(n_sel), _ptr(sel_jobs),
                 C.pointer(n_asg), _ptr(a_job), _ptr(a_off), _ptr(a_w))
        self._check(self.lib.swb_gavel_round(self.h, C.byref(a)), "swb_gavel_round")
        sel = {int(type_order[ti]): sel_jobs[ti, :n_sel[ti]].tolist() for ti in range(W)}
        asg = [(int(a_job[s]), tuple(a_w[a_off[s]:a_off[s + 1]].tolist())) for s in range(n_asg.value)]
        return prio, sel, asg

    def job_table_stats(self):
        used, holes = C.c_int64(), C.c_int64()
        self._check(self.lib.swb_job_table_stats(self.h, C.byref(used), C.byref(holes)), "swb_job_table_stats")
        return dict(used_rows=used.value, hole_rows=holes.value)

    def _round_args(self, slots, progress, meas_ns, meas_end, reestimate, grd):
        slots = np.ascontiguousarray(slots, dtype=np.int32)
        progress = np.ascontiguousarray(progress, dtype=np.int32)
        meas_ns = np.ascontiguousarray(meas_ns, dtype=np.float64)
        meas_end = np.ascontiguousarray(meas_end, dtype=np.int32)
        a = RoundArgs()
        a.J, a.reestimate_share, a.gavel_round_duration = len(slots), int(bool(reestimate)), float(grd)
        a.slots, a.epoch_progress, a.meas_nsamples, a.meas_end_round = _ptr(slots), _ptr(progress), _ptr(meas_ns), _ptr(meas_end)
        return a, (slots, progress, meas_ns, meas_end)

    def round_solve(self, params, slots, progress, meas_ns, meas_end, reestimate, grd, want_forecast=False,
                    packed=False):
        """packed=True: x / backfill come back as [J, 2] uint64 round masks (`xmask`, `bfmask`) instead of J x T bytes."""
        a, keep = self._round_args(slots, progress, meas_ns, meas_end, reestimate, grd)
        J, T = a.J, params.future_rounds
        x = bf = xm = bm = None
        if packed:
            xm = np.empty((J, 2), dtype=np.uint64); bm = np.empty((J, 2), dtype=np.uint64)
        else:
            x = np.zeros((J, T), dtype=np.uint8); bf = np.zeros((J, T), dtype=np.uint8)
        nr = np.empty(J, dtype=np.int32)
        fo = np.empty((6, J), dtype=np.float64) if want_forecast else None
        res = Result()
        a.x, a.backfill, a.nrounds, a.forecast_out, a.res = _ptr(x), _ptr(bf), _ptr(nr), _ptr(fo), C.pointer(res)
        a.xmask, a.bfmask = _ptr(xm), _ptr(bm)
        self._check(self.lib.swb_round_solve(self.h, C.byref(params), C.byref(a)), "swb_round_solve")
        out = dict(x=x, backfill=bf, xmask=xm, bfmask=bm, nrounds=nr, result=res.as_dict())
        if want_forecast:
            fb = res.status == ST_FALLBACK
            out.update(dbar=fo[0], rem=fo[1], ftobj=fo[2], bfkey=fo[5] if fb else fo[3], rem_fb=fo[4])
        return out

    def forecast(self, params, slots, progress, meas_ns, meas_end, reestimate, grd):
        a, keep = self._round_args(slots, progress, meas_ns, meas_end, reestimate, grd)
        J = a.J
        outs = [np.zeros(J, dtype=np.float64) for _ in range(5)]
        self._check(self.lib.swb_forecast(self.h, C.byref(params), C.byref(a), *[_ptr(o) for o in outs]),
                    "swb_forecast")
        return dict(dbar=outs[0], rem=outs[1], ftobj=outs[2], bfkey=outs[3], ft_estimate=outs[4])

    def forecast_commit(self, fallback, ncal):
        ncal = np.ascontiguousarray(ncal, dtype=np.int32)
        self._check(self.lib.swb_forecast_commit(self.h, len(ncal), int(bool(fallback)), _ptr(ncal)),
                    "swb_forecast_commit")

    def sync(self):
        """Wait for everything queued on the context's stream (needed after calls made under OPT_ASYNC_AUX)."""
        self._check(self.lib.swb_sync(self.h), "swb_sync")

    def set_option(self, option, value):
        self._check(self.lib.swb_set_option(self.h, int(option), int(value)), "swb_set_option")

    def allox_assign(self, p, t, wtype):
        """min-cost assignment of m jobs to (worker, position) columns; p [m, W], t [m], wtype [n] int."""
        p = np.ascontiguousarray(p, dtype=np.float64); t = np.ascontiguousarray(t, dtype=np.float64)
        wtype = np.ascontiguousarray(wtype, dtype=np.int32)
        m, W = p.shape
        n = len(wtype)
        cols = np.zeros(m, dtype=np.int32)
        tot = C.c_double()
        self._check(self.lib.swb_allox_assign(self.h, m, n, W, _ptr(p), _ptr(t), _ptr(wtype), _ptr(cols),
                                              C.byref(tot)), "swb_allox_assign")
        return cols, tot.value

    def lp_solve(self, colp, rowi, val, c, b, max_iter=0):
        """Batch of S linear programs  max c'x : A x <= b, x >= 0  with a shared CSC pattern (swb_lp_solve).
        colp [n+1], rowi [nnz] int32; val [S, nnz], c [S, n], b [S, m] float64 (1-D arrays mean S = 1).
        Returns x [S, n], objective [S], status [S], stats [S, 4]."""
        colp = np.ascontiguousarray(colp, dtype=np.int32); rowi = np.ascontiguousarray(rowi, dtype=np.int32)
        val = np.atleast_2d(np.ascontiguousarray(val, dtype=np.float64))
        c = np.atleast_2d(np.ascontiguousarray(c, dtype=np.float64))
        b = np.atleast_2d(np.ascontiguousarray(b, dtype=np.float64))
        S, n = c.shape
        m = b.shape[1]
        nnz = len(rowi)
        if val.shape != (S, nnz) or b.shape[0] != S or len(colp) != n + 1:
            raise ValueError("lp_solve: inconsistent array shapes")
        x = np.zeros((S, n)); obj = np.zeros(S); status = np.zeros(S, dtype=np.int32)
        stats = np.zeros((S, 4), dtype=np.int32)
        if max_iter <= 0:
            max_iter = 50 * (m + n) + 1000
        self._check(self.lib.swb_lp_solve(self.h, S, m, n, nnz, _ptr(colp), _ptr(rowi), _ptr(val), _ptr(c), _ptr(b),
                                          int(max_iter), _ptr(x), _ptr(obj), _ptr(status), _ptr(stats)),
                    "swb_lp_solve")
        return x, obj, status, stats

    def last_timings(self):
        a, b, n = C.c_double(), C.c_double(), C.c_int32()
        self._check(self.lib.swb_last_timings(self.h, C.byref(a), C.byref(b), C.byref(n)), "swb_last_timings")
        return dict(ms_solve=a.value, ms_place=b.value, passes=n.value)

    def stream_ptr(self):
        return int(self.lib.swb_stream(self.h) or 0)

    def gbm_forecast_device(self, J, R0_ptr, H_ptr, mu_ptr, sigma_ptr, P_local, path_offset, seed, out_ptr):
        """All-device variant: raw device pointers in, partial sums written to out_ptr ([2, J] float64)."""
        vp = lambda v: C.c_void_p(int(v))
        self._check(self.lib.swb_gbm_forecast(self.h, int(J), vp(R0_ptr), vp(H_ptr), vp(mu_ptr), vp(sigma_ptr),
                                              int(P_local), int(path_offset), int(seed), vp(out_ptr), 3),
                    "swb_gbm_forecast")

    def gbm_forecast(self, R0, H, mu, sigma, P_local, path_offset=0, seed=0, out_device_ptr=None):
        """Sums over the local sample paths: returns [2, J] (host) or writes them to `out_device_ptr`."""
        R0 = np.ascontiguousarray(R0, dtype=np.float64); mu = np.ascontiguousarray(mu, dtype=np.float64)
        sigma = np.ascontiguousarray(sigma, dtype=np.float64); H = np.ascontiguousarray(H, dtype=np.int32)
        J = len(R0)
        if out_device_ptr:
            self._check(self.lib.swb_gbm_forecast(self.h, J, _ptr(R0), _ptr(H), _ptr(mu), _ptr(sigma), int(P_local),
                                                  int(path_offset), int(seed), C.c_void_p(int(out_device_ptr)), 1),
                        "swb_gbm_forecast")
            return None
        out = np.zeros((2, J), dtype=np.float64)
        self._check(self.lib.swb_gbm_forecast(self.h, J, _ptr(R0), _ptr(H), _ptr(mu), _ptr(sigma), int(P_local),
                                              int(path_offset), int(seed), _ptr(out), 0), "swb_gbm_forecast")
        return out


def market_pgd(eng, params, g, E, c, dbar, rem, rate, Gw, X, iters, coarse_iters=0, primal_weight=0.0, cap=None,
               warm_start=False, device_ptrs=None, utility=0):
    """Dense primal-dual price-response iterations on X[S,J,W,T] (fp32): `coarse_iters` on the time-coarsened tensor,
    then `iters` on the full one.  Host arrays by default (X is overwritten with the feasible result; its content is
    the starting point only with warm_start); `device_ptrs` = dict(g,E,c,dbar,rem,rate,X) of raw device pointers for
    resident data.  Gw [W] workers per type, or cap [W,T] workers per type and round.
    Returns (obj[S,3] = objective, makespan, capacity violation before the final repair ; ms of the last dense pass)."""
    lib = eng.lib
    plist = params if isinstance(params, (list, tuple)) else [params]
    S = len(plist)
    a = MarketArgs()
    obj = np.zeros((S, 3), dtype=np.float64)
    ms = C.c_float()
    a.iters, a.coarse_iters, a.warm_start = int(iters), int(coarse_iters), int(bool(warm_start))
    a.primal_weight = float(primal_weight)
    a.utility = int(utility)
    a.prm = (Params * S)(*plist)
    if cap is not None:
        cap = np.ascontiguousarray(cap, dtype=np.float64)
        a.cap = _ptr(cap)
    if Gw is not None:
        Gw = np.ascontiguousarray(Gw, dtype=np.float64)
        a.Gw = _ptr(Gw)
    a.obj, a.dense_ms = _ptr(obj), C.pointer(ms)
    if device_ptrs is None:
        g = np.ascontiguousarray(g, dtype=np.int32)
        f64 = lambda v: np.ascontiguousarray(v, dtype=np.float64)
        E, c, dbar, rem = f64(E), f64(c), f64(dbar), f64(rem)
        rate = np.ascontiguousarray(rate, dtype=np.float32)
        assert X.dtype == np.float32 and X.flags.c_contiguous and X.ndim == 4
        a.S, a.J, a.W, a.T = X.shape
        a.per_scenario_jobs, a.on_device = (1 if g.ndim == 2 else 0), 0
        a.g, a.E, a.c, a.dbar, a.rem, a.rate, a.X = _ptr(g), _ptr(E), _ptr(c), _ptr(dbar), _ptr(rem), _ptr(rate), _ptr(X)
        keep = (g, E, c, dbar, rem, rate)
    else:
        a.S, a.J, a.W, a.T = device_ptrs["shape"]
        a.per_scenario_jobs, a.on_device = int(device_ptrs.get("per_scenario_jobs", 0)), 1
        vp = lambda k: C.c_void_p(int(device_ptrs[k]))
        a.g, a.E, a.c, a.dbar, a.rem, a.rate, a.X = vp("g"), vp("E"), vp("c"), vp("dbar"), vp("rem"), vp("rate"), vp("X")
    if cap is not None:
        assert cap.shape == (a.W, a.T)
    rc = lib.swb_market_pgd(eng.h, C.byref(a))
    if rc < 0:
        raise RuntimeError(f"swb_market_pgd failed ({rc}): {lib.swb_last_error().decode()}")
    return obj, float(ms.value)
