"""What-if ensembles of a trace on the device (SURVEY §8(f)-4): the round loop of the reference simulator
(`Scheduler.simulate()` scheduler/scheduler.py:1878-2250) as `swb_sim_*` (csrc/sim.cu) — time advance, progress,
preemption overhead, retirement, arrivals and the measured-throughput timeline of S scenarios per launch — with the
policy of every scenario deciding between two steps:

* `DeviceSim`            ctypes binding of swb_sim_* (begin / step / replay / results);
* `ShockwaveEnsemble`    S `ShockwaveScheduler` what-ifs (k, lambda, rhomax, future rounds ... per scenario) of one trace
                          in lock-step: per round ONE step launch for all scenarios + one `round_schedule()` per
                          scenario; the per-job Python of the reference's loop (`_done_callback`, `_update_throughput`,
                          `_update_shockwave_scheduler`: O(jobs) dict work per round) is replaced by array updates taken
                          from the step's outputs (`ShockwaveScheduler.schedule_progress_batch`).

One worker type, single jobs (no packing).  Dynamic adaptation (accordion / gns batch-size rescaling) runs from
tables: `build_dynamic_tables` lays them out from the reference's rules, the throughput file and the reference's own
gns pattern generator (see INTEGRATION.md).
No CPU path: the binding raises when libswb200.so or the GPU is missing."""
import ctypes as C
import math
from collections import OrderedDict

import numpy as np

from . import engine as _eng
from .engine import SCN_DTYPE, SimDynamic, SimTrace
from .scheduler import ShockwaveScheduler

REOPT_ROUNDS = 8          # scheduler/scheduler.py:71


def pack_dynamic_tables(dyn, J):
    """build_dynamic_tables() output -> the flat arrays of swb_sim_dynamic (kept alive by the returned dict)."""
    K = max(1, max(len(v) for v in dyn["lvl_bs"]))
    if K > MAX_LEVELS:
        raise ValueError("more than 8 batch-size levels for one job")
    a = {k: np.ascontiguousarray(dyn[k], dtype=np.int32) for k in ("mode", "bs_max", "bs_min", "bs_big", "orig_locked", "acc_skip")}
    off = np.zeros(J + 1, np.int64)
    off[1:] = np.cumsum([len(p) for p in dyn["pattern"]])
    a["pat_off"] = off
    a["pattern"] = np.ascontiguousarray(np.concatenate([np.asarray(p, np.int32) for p in dyn["pattern"]] + [np.zeros(1, np.int32)]))
    lb = np.zeros((J, K), np.int32)
    lt = np.zeros((J, K), np.float64)
    for j in range(J):
        n = len(dyn["lvl_bs"][j])
        lb[j, :n] = dyn["lvl_bs"][j]
        lt[j, :n] = dyn["lvl_thr"][j]
    a["lvl_bs"], a["lvl_thr"], a["K"] = lb, lt, K
    return a


TRACE_KEYS = (("arrival", np.float64), ("total_steps", np.int64), ("scale_factor", np.int32), ("throughput", np.float64),
              ("duration", np.float64), ("batch_size", np.int32), ("dataset_len", np.int64))


class DeviceSim:
    """swb_sim_*: S scenarios of one static trace.  trace: dict of [J] sequences (TRACE_KEYS) + optional
    `adaptation_mode` ([J] int, 0 = static)."""

    def __init__(self, trace, S, ngpus, time_per_iteration=120.0, round_duration=None, device=0):
        self._lib = _eng.load_library()
        self._h = None
        self.S, self.J = int(S), len(trace["arrival"])
        self._arr = {k: np.ascontiguousarray(trace[k], dtype=dt) for k, dt in TRACE_KEYS}
        for k, a in self._arr.items():
            if a.shape != (self.J,):
                raise ValueError(f"trace[{k!r}] must have one entry per job")
        t = SimTrace()
        t.J = self.J
        for k, _ in TRACE_KEYS:
            setattr(t, k, self._arr[k].ctypes.data)
        if trace.get("adaptation_mode") is not None:
            self._arr["adaptation_mode"] = np.ascontiguousarray(trace["adaptation_mode"], dtype=np.int32)
            t.adaptation_mode = self._arr["adaptation_mode"].ctypes.data
        h = C.c_void_p()
        rd = time_per_iteration if round_duration is None else round_duration
        self._ck(self._lib.swb_sim_create(int(device), C.byref(t), self.S, int(ngpus), float(time_per_iteration),
                                          float(rd), C.byref(h)))
        self._h = h
        S, J = self.S, self.J
        self.scn = np.zeros(S, dtype=SCN_DTYPE)
        self.status = np.zeros((S, J), np.uint8)
        self.epoch = np.zeros((S, J), np.int32)
        self.tl_ns = np.zeros((S, J), np.float64)
        self.tl_end = np.full((S, J), -1, np.int32)

    def _ck(self, rc):
        if rc != 0:
            raise RuntimeError(f"libswb200: {self._lib.swb_last_error().decode()} (code {rc})")

    def set_dynamic(self, dyn):
        """dyn: build_dynamic_tables() output (accordion / gns jobs)."""
        a = pack_dynamic_tables(dyn, self.J)
        d = SimDynamic()
        for k in ("mode", "bs_max", "bs_min", "bs_big", "orig_locked", "acc_skip", "pat_off", "pattern", "lvl_bs", "lvl_thr"):
            setattr(d, k, a[k].ctypes.data)
        d.n_levels = a["K"]
        self._ck(self._lib.swb_sim_set_dynamic(self._h, C.byref(d)))

    def set_worker_types(self, throughput, ngpus):
        """Several worker types (static jobs): throughput [J][W] (`Scheduler._throughputs[job][worker_type]`, 0 = the
        job cannot run there), ngpus [W].  Afterwards chosen[s][j] = 1 + index of the type job j runs on."""
        thr = np.ascontiguousarray(throughput, dtype=np.float64)
        cap = np.ascontiguousarray(ngpus, dtype=np.int32)
        if thr.ndim != 2 or thr.shape != (self.J, cap.shape[0]):
            raise ValueError("throughput must be [J][W] and ngpus [W]")
        self._ck(self._lib.swb_sim_set_worker_types(self._h, int(cap.shape[0]), thr.ctypes.data, cap.ctypes.data))
        self.W = int(cap.shape[0])

    def begin(self):
        self._ck(self._lib.swb_sim_begin(self._h, self.scn.ctypes.data, self.status.ctypes.data))
        return self.scn

    def step(self, chosen):
        ch = np.ascontiguousarray(chosen, dtype=np.uint8)
        if ch.shape != (self.S, self.J):
            raise ValueError("chosen must be [S][J]")
        self._ck(self._lib.swb_sim_step(self._h, ch.ctypes.data, self.scn.ctypes.data, self.status.ctypes.data,
                                        self.epoch.ctypes.data, self.tl_ns.ctypes.data, self.tl_end.ctypes.data))
        return self.scn

    def replay(self, schedule):
        """schedule [R][J] (shared) or [R][S][J]: begin + all rounds in one launch."""
        sc = np.ascontiguousarray(schedule, dtype=np.uint8)
        if sc.ndim == 2 and sc.shape[1] == self.J:
            per = 0
        elif sc.ndim == 3 and sc.shape[1:] == (self.S, self.J):
            per = 1
        else:
            raise ValueError("schedule must be [R][J] or [R][S][J]")
        self._ck(self._lib.swb_sim_replay(self._h, sc.ctypes.data, sc.shape[0], per, self.scn.ctypes.data))
        return self.scn

    def results(self):
        S, J = self.S, self.J
        jct = np.zeros((S, J)); steps = np.zeros((S, J), np.int64); rt = np.zeros((S, J)); tm = np.zeros((S, J))
        self._ck(self._lib.swb_sim_results(self._h, jct.ctypes.data, steps.ctypes.data, rt.ctypes.data, tm.ctypes.data))
        return dict(jct=jct, steps_run=steps, run_time=rt, measured_throughput=tm)

    def job_state(self):
        """Current total steps / throughput / batch size, execution and finish time of the latest round, failed attempts in
        a row, ran-in-the-latest-round flag: [S][J] each (swb_sim_job_state)."""
        S, J = self.S, self.J
        out = dict(total_steps=np.zeros((S, J), np.int64), throughput=np.zeros((S, J)), batch_size=np.zeros((S, J), np.int32),
                   exec_time=np.zeros((S, J)), finish_time=np.zeros((S, J)), failed_attempts=np.zeros((S, J), np.uint8),
                   ran=np.zeros((S, J), np.uint8))
        self._ck(self._lib.swb_sim_job_state(self._h, *[out[k].ctypes.data for k in (
            "total_steps", "throughput", "batch_size", "exec_time", "finish_time", "failed_attempts", "ran")]))
        return out

    def close(self):
        if self._h is not None:
            self._lib.swb_sim_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class TraceJob:
    """What ShockwaveScheduler reads of a job (the attribute surface of the reference's JobMetaData,
    scheduler/JobMetaData.py:40-110), built from the reference's profile dict (utils.generate_pickle_file)."""

    def __init__(self, jobid, profile, round_duration, overclock=1.0):
        self.jobid = jobid
        self.nworkers = int(profile.get("scale_factor", 1))
        self.epochs = int(profile["num_epochs"])
        self.epoch_nsamples = profile["num_samples_per_epoch"]
        dur = [max(1.0, round(d)) for d in profile["duration_every_epoch"]]        # JobMetaData.py:112-115
        dur = [max(1.0, d / float(overclock)) for d in dur]                         # :117-121
        assert len(dur) == self.epochs
        self.epoch_duration = dur
        self.epoch_duration_preprofiled = list(dur)
        self.bs_schedule = list(profile["bs_every_epoch"])
        assert len(self.bs_schedule) == self.epochs
        self.throughput_measurements = OrderedDict()    # stays empty: the summaries come from the device step
        self.gavel_round_duration = round_duration
        self.epoch_progress = 0
        self.timestamp_submit = None
        self.waiting_delay = 0

    def set_epoch_progress(self, p):
        assert 0 <= p <= self.epochs
        self.epoch_progress = p

    def add_waiting_delay(self, d):
        self.waiting_delay += d

    def reset_waiting_delay(self):
        self.waiting_delay = 0


class ShockwaveEnsemble:
    """S Shockwave what-ifs of one static trace.  `scenarios`: list of dicts overriding `config` (the reference's
    shockwave_config json keys: future_rounds, k, lambda, rhomax, log_approximation_bases, ...) per scenario."""

    def __init__(self, trace, profiles, config, scenarios, ngpus, time_per_iteration=120, device=0,
                 scheduler_kwargs=None, dynamic=None):
        if float(trace["arrival"][0]) != 0.0:
            # the reference's loop iterates `_scheduled_jobs_in_current_round = None` when the first round does not
            # start at t = 0 (scheduler.py:359, :2273-2277): its shockwave traces all start at 0
            raise ValueError("the first job of a shockwave trace must arrive at t = 0")
        self.trace, self.profiles, self.ngpus = trace, profiles, int(ngpus)
        self.tpi = time_per_iteration
        self.S, self.J = len(scenarios), len(trace["arrival"])
        self.sim = DeviceSim(trace, self.S, ngpus, time_per_iteration, time_per_iteration, device)
        if dynamic is not None:                      # build_dynamic_tables(): accordion / gns jobs
            self.sim.set_dynamic(dynamic)
        self.scheds = []
        for ov in scenarios:
            cfg = dict(config)
            cfg.update(ov)
            bases = cfg["log_approximation_bases"]
            origin = cfg.get("log_approximation_origin", {0.0: 1e-6})
            origin = {float(k): v for k, v in origin.items()}
            self.scheds.append(ShockwaveScheduler(
                ngpus=self.ngpus, gram=cfg.get("gpu_ram", 32), init_metadata=OrderedDict(),
                future_nrounds=cfg["future_rounds"], round_duration=time_per_iteration,
                solver_preference=cfg.get("solver_preference", ["GUROBI"]), solver_rel_gap=cfg.get("solver_rel_gap", 1e-3),
                solver_num_threads=cfg.get("solver_num_threads", 1), solver_timeout=cfg.get("solver_timeout", 15),
                n_epoch_vars_max=max(cfg["future_rounds"], 30), logapx_bases=bases, logapx_origin=origin,
                k=cfg["k"], lam=cfg["lambda"], rhomax=cfg["rhomax"], device=device, **(scheduler_kwargs or {})))
        self.per_round_schedule = [[] for _ in range(self.S)]
        self.resolves = np.zeros(self.S, np.int64)

    def run(self, max_rounds=None, threads=None):
        """threads: host threads the per-scenario scheduler calls of one round are spread over (default min(S, 8), 0 or 1
        = serial).  Every scenario owns its scheduler, context and stream and ctypes drops the GIL inside the C call, so
        the re-solves of different scenarios overlap on the GPU; results do not depend on it."""
        sim, S, J = self.sim, self.S, self.J
        scn = sim.begin()
        status = sim.status.copy()
        live_prev = np.zeros((S, J), bool)
        chosen_prev = np.zeros((S, J), np.uint8)
        ireopt = [0] * S
        nthreads = min(S, 8) if threads is None else int(threads)
        pool = None
        if nthreads > 1:
            from concurrent.futures import ThreadPoolExecutor
            pool = ThreadPoolExecutor(max_workers=nthreads)
        c = 0

        def one(s):
            sch = self.scheds[s]
            live = status[s] == 1
            if c > 0 and scn["now"][s] != 0.0:
                # _update_shockwave_scheduler (scheduler.py:2270-2375) for the round that just ended
                ran = np.flatnonzero((chosen_prev[s] == 1) & live)
                sch.schedule_progress_batch(ran.tolist(), sim.epoch[s, ran], sim.tl_ns[s, ran], sim.tl_end[s, ran])
                sch.increment_round_ptr()
                ireopt[s] += 1
                if ireopt[s] >= REOPT_ROUNDS:
                    ireopt[s] = 0
                    sch.set_resolve()
            for j in np.flatnonzero(live_prev[s] & ~live).tolist():        # _remove_job -> remove_metadata
                sch.remove_metadata(j)
            for j in np.flatnonzero(live & ~live_prev[s]).tolist():        # add_job -> add_metadata
                job = TraceJob(j, self.profiles[j], self.tpi)
                job.timestamp_submit = float(scn["now"][s])                 # register_job_submit(current timestamp)
                sch.add_metadata(j, job)
            live_prev[s] = live
            was = sch.resolve
            ids = sch.round_schedule()
            self.resolves[s] += bool(was)
            return [j for j in ids if live[j]]

        while not scn["done"].all():
            chosen = np.zeros((S, J), np.uint8)
            todo = [s for s in range(S) if not scn["done"][s]]
            picked = list(pool.map(one, todo)) if pool is not None else [one(s) for s in todo]
            for s, ids in zip(todo, picked):
                chosen[s, ids] = 1
                self.per_round_schedule[s].append(sorted(ids))
            scn = sim.step(chosen)
            if (scn["err"] != 0).any():
                raise RuntimeError(f"swb_sim_step: error flags {scn['err'].tolist()}")
            status = sim.status.copy()
            chosen_prev = chosen
            c += 1
            if max_rounds is not None and c >= max_rounds:
                break
        if pool is not None:
            pool.shutdown()
        res = sim.results()
        res.update(makespan=scn["now"].copy(), rounds=scn["rounds"].copy(), per_round_schedule=self.per_round_schedule,
                   resolves=self.resolves.copy(), avg_jct=np.nanmean(res["jct"], axis=1))
        self.last = res
        return res

    def result_dicts(self, res=None, trace_file=None):
        """One dict per scenario with the keys of the result pickle `simulate_scheduler_with_trace.py` writes
        (scripts/drivers/simulate_scheduler_with_trace.py:128-151), so `aggregate_result.py` / `plotting.py` can read
        what a sweep produced.  Filled: makespan, avg_jct, geometric / harmonic mean (scheduler.py:2779-2840),
        jct_list, finish_time_fairness_list (:2865-2925: completion time / (isolated run time x max(1, jobs / GPUs)),
        rounded to 5 digits), cluster_util (GPU-seconds used / (GPUs x makespan): the mean of the reference's per-worker
        figures before its per-worker rounding), per_round_schedule (job ids per round; no worker ids), job_run_time,
        time_per_iteration.  Absent: everything that needs worker identities (utilization_list, envy lists, lease
        extension counts) — the device loop does not assign worker ids."""
        res = self.last if res is None else res
        J = self.J
        iso = np.array([sum(p["duration_every_epoch"]) for p in self.profiles[:J]], dtype=np.float64)
        contention = max(1.0, J / self.ngpus)
        sf = np.asarray(self.trace["scale_factor"], dtype=np.float64)
        out = []
        for s in range(self.S):
            jct = res["jct"][s]
            done = np.isfinite(jct)
            jl = [float(v) for v in jct[done]]
            ftf = [round(float(jct[j]) / (float(iso[j]) * contention), 5) for j in range(J) if done[j]]
            out.append({
                "trace_file": trace_file, "policy": "shockwave", "scenario": s,
                "makespan": float(res["makespan"][s]), "avg_jct": float(np.mean(jl)) if jl else None,
                "geometric_mean_jct": float(np.exp(np.mean(np.log(jl)))) if jl else None,
                "harmonic_mean_jct": float(len(jl) / np.sum(1.0 / np.asarray(jl))) if jl else None,
                "jct_list": jl, "finish_time_fairness_list": ftf,
                "cluster_util": float((sf * res["run_time"][s]).sum() / (self.ngpus * res["makespan"][s])),
                "per_round_schedule": [{j: None for j in rnd} for rnd in res["per_round_schedule"][s]],
                "job_run_time": {j: float(res["run_time"][s, j]) for j in range(J)},
                "time_per_iteration": self.tpi})
        return out

    def write_result_pickles(self, directory, res=None, trace_file=None, prefix="shockwave_scenario"):
        import os
        import pickle
        os.makedirs(directory, exist_ok=True)
        paths = []
        for d in self.result_dicts(res, trace_file):
            path = os.path.join(directory, f"{prefix}_{d['scenario']}.pickle")
            with open(path, "wb") as f:
                pickle.dump(d, f)
            paths.append(path)
        return paths


# ---- dynamic adaptation (accordion / gns batch-size rescaling) as tables -------------------------------------------
# The reference decides rescale requests from per-model rules hard-wired into its simulator.  The device loop takes
# them as tables; this builder lays the tables out from the same rules (constants cited line by line) plus two things
# only the caller has: the throughput file and the reference's own gns pattern generator.
AT_MAX_BS = {"ResNet-18": 256, "ResNet-50": 128, "Transformer": 128, "LM": 80, "Recommendation": 8192}   # scheduler.py:1636-1646
AT_MIN_BS = {"ResNet-18": 16, "ResNet-50": 16, "Transformer": 16, "LM": 5, "Recommendation": 512}       # scheduler.py:1711-1721
MAX_BS_DICT = {"LM": 80, "ResNet-18": 256, "ResNet-50": 128, "Recommendation": 8192}                    # scheduler.py:4756-4761
MODE_CODE = {"static": 0, "accordion": 1, "gns": 2}
GNS_PATTERN_EPOCHS = 760                                                                                # scheduler.py:1619
MAX_LEVELS = 8


def accordion_critical(model, original_bs, epoch):
    """in_critical_regime of _simulate_accordion (scheduler.py:1670-1692); None where the reference leaves it unset."""
    if model == "LM":
        return epoch < 10
    if model == "Recommendation":
        if original_bs in (512, 1024):
            return epoch < 30
        if original_bs == 2048:
            return epoch < 40
        if original_bs in (4096, 8192):
            return epoch < 10
        return None
    if model == "ResNet-50":
        return (epoch % 30) < 10
    if model == "ResNet-18":
        head = 20 if original_bs == 256 else 10
        return (0 <= epoch < head) or (150 <= epoch < 160) or (250 <= epoch < 260)
    return None


def build_dynamic_tables(models, modes, trace, throughput_of, gns_pattern):
    """Tables for swb_sim_set_dynamic.  models[j]: "ResNet-18", "LM", ...; modes[j]: "static" / "accordion" / "gns";
    trace: the static arrays (batch_size = ORIGINAL batch size, total_steps, dataset_len, scale_factor);
    throughput_of(model, batch_size, scale_factor) -> steps/s on the worker type or None when the throughput file has no
    such entry; gns_pattern(job_type, batch_size, num_epochs, scale_factor) -> list: the reference's
    utils.get_gns_bs_pattern (scheduler/utils.py:801-1010), called exactly as _simulate_gns does."""
    J = len(models)
    out = dict(mode=np.zeros(J, np.int32), bs_max=np.zeros(J, np.int32), bs_min=np.zeros(J, np.int32),
               bs_big=np.full(J, -1, np.int32), orig_locked=np.zeros(J, np.int32), acc_skip=np.zeros(J, np.int32),
               pattern=[], lvl_bs=[], lvl_thr=[])
    for j in range(J):
        model, bs0, sf = models[j], int(trace["batch_size"][j]), int(trace["scale_factor"][j])
        mode = MODE_CODE[modes[j]]
        out["mode"][j] = mode
        out["bs_max"][j] = AT_MAX_BS.get(model, -1)
        out["bs_min"][j] = AT_MIN_BS.get(model, -1)
        out["bs_big"][j] = MAX_BS_DICT.get(model, -1)
        out["orig_locked"][j] = int(model in MAX_BS_DICT and bs0 == MAX_BS_DICT[model])      # scheduler.py:4767-4775
        cand = sorted({bs0 * (1 << i) for i in range(MAX_LEVELS)} | ({MAX_BS_DICT[model]} if model in MAX_BS_DICT else set()))
        lv = [(b, throughput_of(model, b, sf)) for b in cand]
        lv = [(b, t) for b, t in lv if t is not None][:MAX_LEVELS]
        out["lvl_bs"].append([b for b, _ in lv])
        out["lvl_thr"].append([float(t) for _, t in lv])
        if mode == 1:
            out["acc_skip"][j] = int(model == "Transformer")                                  # scheduler.py:1667-1669
            spe = math.ceil(int(trace["dataset_len"][j]) / bs0)
            n = math.ceil(int(trace["total_steps"][j]) / spe) + 8
            crit = [accordion_critical(model, bs0, e) for e in range(n)]
            if not out["acc_skip"][j] and any(v is None for v in crit):
                raise ValueError(f"job {j}: the reference has no accordion rule for {model} at batch size {bs0}")
            out["pattern"].append([int(bool(v)) for v in crit])
        elif mode == 2:
            # _simulate_gns asks for max(760, epoch + 2) epochs and reads entries epoch and epoch + 1 (:1617-1632).  The
            # generator never scales the LAST entry of what it returns, every other entry does not depend on the length:
            # one long table + the rule "entry epoch + 1 is the original batch size once epoch + 1 >= 759" (sim_core.cuh)
            spe = math.ceil(int(trace["dataset_len"][j]) / bs0)
            n = max(GNS_PATTERN_EPOCHS + 2, math.ceil(int(trace["total_steps"][j]) / spe) + 8)
            out["pattern"].append([int(v) for v in gns_pattern(f"{model} (batch size {bs0})", bs0, n, sf)])
        else:
            out["pattern"].append([])
    return out


# ---- several GPUs: what-if scenarios are independent, so they shard with no data-path collective ----------------------
def shard_scenarios(n_scenarios, rank, world):
    """Indices of the scenarios rank `rank` runs (round-robin: neighbouring sweep points usually cost alike)."""
    return list(range(rank, n_scenarios, world))


def run_sharded(trace, profiles, config, scenarios, ngpus, rank=0, world=1, gather=None, device=None, **kw):
    """One process per GPU: every rank runs ShockwaveEnsemble on its slice of `scenarios` (device = its GPU), then the
    small per-scenario results are exchanged with `gather` (e.g. `lambda obj: all_gather_object(...)` over NCCL/gloo —
    results only, nothing on the data path).  Returns, on every rank, the result dict in the ORIGINAL scenario order."""
    mine = shard_scenarios(len(scenarios), rank, world)
    part = None
    if mine:
        ens = ShockwaveEnsemble(trace, profiles, config, [scenarios[i] for i in mine], ngpus,
                                device=rank if device is None else device, **kw)
        r = ens.run()
        part = dict(index=mine, makespan=r["makespan"], rounds=r["rounds"], jct=r["jct"], avg_jct=r["avg_jct"],
                    resolves=r["resolves"], per_round_schedule=r["per_round_schedule"], run_time=r["run_time"])
    parts = [part] if gather is None else gather(part)
    S, J = len(scenarios), len(trace["arrival"])
    out = dict(makespan=np.full(S, np.nan), rounds=np.zeros(S, np.int64), jct=np.full((S, J), np.nan),
               avg_jct=np.full(S, np.nan), resolves=np.zeros(S, np.int64), per_round_schedule=[None] * S,
               run_time=np.zeros((S, J)))
    for p in parts:
        if p is None:
            continue
        for k, i in enumerate(p["index"]):
            for key in ("makespan", "rounds", "jct", "avg_jct", "resolves", "run_time"):
                out[key][i] = p[key][k]
            out["per_round_schedule"][i] = p["per_round_schedule"][k]
    return out


def run_policies_sharded(trace, policy_names, ngpus, rank=0, world=1, gather=None, device=None, make_policy=None, **kw):
    """The Gavel-policy counterpart of run_sharded: every rank runs PolicyEnsemble on its round-robin slice of
    `policy_names` (what-ifs = policies, one per scenario; the policy kernels and the round step run on the rank's GPU),
    then only the per-scenario results travel through `gather`.  make_policy(name) builds one policy object (default:
    `policies.get_policy(name, solver="ECOS")`); **kw goes to PolicyEnsemble (dynamic=, worker_types=, ...).  Returns, on
    every rank, the result dict in the ORIGINAL order."""
    from . import policies as _pol
    mine = shard_scenarios(len(policy_names), rank, world)
    dev = rank if device is None else device
    part = None
    if mine:
        _pol.set_device(dev)
        mk = make_policy or (lambda n: _pol.get_policy(n, solver="ECOS", seed=0))
        ens = PolicyEnsemble(trace, [mk(policy_names[i]) for i in mine], ngpus, device=dev, **kw)
        r = ens.run()
        part = dict(index=mine, makespan=r["makespan"], rounds=r["rounds"], jct=r["jct"], avg_jct=r["avg_jct"],
                    allocations=r["allocations"], per_round_schedule=r["per_round_schedule"], run_time=r["run_time"])
    parts = [part] if gather is None else gather(part)
    S, J = len(policy_names), len(trace["arrival"])
    out = dict(makespan=np.full(S, np.nan), rounds=np.zeros(S, np.int64), jct=np.full((S, J), np.nan),
               avg_jct=np.full(S, np.nan), allocations=np.zeros(S, np.int64), per_round_schedule=[None] * S,
               run_time=np.zeros((S, J)))
    for p in parts:
        if p is None:
            continue
        for k, i in enumerate(p["index"]):
            for key in ("makespan", "rounds", "jct", "avg_jct", "allocations", "run_time"):
                out[key][i] = p[key][k]
            out["per_round_schedule"][i] = p["per_round_schedule"][k]
    return out


# ---- Gavel policies on the device loop -----------------------------------------------------------------------------------
class PolicyEnsemble:
    """S what-ifs of one trace under the Gavel policies (one policy object per scenario, e.g.
    `policies.get_policy("max_min_fairness")`, `("finish_time_fairness")`, ...): the round loop runs on the device
    (swb_sim_step), `get_allocation()` and the priority -> selection -> worker-assignment step (swb_gavel_round) are the
    device calls of policies.py / placement.py, and what the reference keeps in dicts between two rounds is kept here in
    arrays, statement by statement:
      * time accounting of `_done_callback` (scheduler.py:4660-4672): `_job_time_so_far`, `_worker_time_so_far`, added in
        the reference's completion order (latest finish first, then job id) so the float sums are the same;
      * `_update_priorities` (:3611-3636): when to reset the accounting and recompute the allocation
        (`_need_to_update_allocation` after an arrival, a completion or a failed micro-task; at most once per
        `minimum_time_between_allocation_resets`), `_reset_time_run_so_far` (:3498-3551) with its deficits;
      * `_get_allocation_state` / `_compute_allocation` (:3205-3355): the arguments each policy family takes.
    Single jobs (no packing).  One worker type by default; `worker_types=dict(names=[...], throughput=[J][W],
    ngpus=[W])` runs a MIXED cluster of static jobs (swb_sim_set_worker_types): names in the reference's sorted order
    (`sorted(cluster_spec)`, scheduler.py:1826 — worker ids are handed out type by type in that order), per-type
    throughputs as in `Scheduler._throughputs[job][worker_type]`; the types are walked in the reference's round order
    v100, p100, k80 (:1290-1301; shuffled by its `_worker_type_shuffler` for policies without "Perf" / "Packing" in
    their name, seed + 5).  Returns per-round schedules WITH worker ids, like the reference."""

    ROUND_ORDER = ("v100", "p100", "k80")              # scheduler.py:1290

    def __init__(self, trace, policies, ngpus, time_per_iteration=120, device=0, dynamic=None, priority_weights=None,
                 minimum_time_between_allocation_resets=1000, round_backend=None, worker_type="v100",
                 other_worker_types=("k80", "p100"), worker_types=None, seed=0):
        self.trace, self.policies, self.tpi = trace, list(policies), time_per_iteration
        self.S, self.J = len(self.policies), len(trace["arrival"])
        if worker_types is not None:
            if dynamic is not None:
                raise ValueError("several worker types run static jobs only")
            self.types = list(worker_types["names"])
            if self.types != sorted(self.types):
                raise ValueError("worker type names must be in sorted order (the reference registers workers that way)")
            self.cap = np.asarray(worker_types["ngpus"], dtype=np.int32)
            self.thr_w = np.ascontiguousarray(worker_types["throughput"], dtype=np.float64)
            if self.thr_w.shape != (self.J, len(self.types)) or self.cap.shape != (len(self.types),) or (self.cap <= 0).any():
                raise ValueError("worker_types: throughput [J][W], ngpus [W] > 0, names [W]")
            ngpus = int(self.cap.sum())
        else:
            self.types, self.cap, self.thr_w = [worker_type], np.array([int(ngpus)], np.int32), None
        self.W = len(self.types)
        self.ngpus = int(ngpus)
        self.sim = DeviceSim(trace, self.S, ngpus, time_per_iteration, time_per_iteration, device)
        if dynamic is not None:
            self.sim.set_dynamic(dynamic)
        if self.thr_w is not None:
            self.sim.set_worker_types(self.thr_w, self.cap)
        self.min_reset = float(minimum_time_between_allocation_resets)
        self.wt = worker_type
        if self.thr_w is not None:
            self.cluster_spec = {w: int(c) for w, c in zip(self.types, self.cap)}
        else:
            self.cluster_spec = {worker_type: self.ngpus, **{w: 0 for w in other_worker_types}}
        import random as _random
        self._shufflers = [_random.Random(seed + 5) for _ in range(self.S)]    # scheduler.py:508-509
        self.pw = np.ones(self.J) if priority_weights is None else np.asarray(priority_weights, dtype=np.float64)
        if round_backend is None:
            from .placement import _DeviceBackend
            round_backend = _DeviceBackend()
        self.backend = round_backend
        self.per_round_schedule = [[] for _ in range(self.S)]
        self.allocations = np.zeros(self.S, np.int64)

    def _allocation(self, s, live, now, st, steps_run):
        """_get_allocation_state + _compute_allocation for scenario s -> alloc [J] (NaN = not in the allocation)."""
        pol, wt = self.policies[s], self.wt
        jobs = np.flatnonzero(live).tolist()
        if self.thr_w is not None:
            thr = {j: {w: float(self.thr_w[j, i]) for i, w in enumerate(self.types)} for j in jobs}
        else:
            thr = {j: {wt: float(st["throughput"][s, j])} for j in jobs}
        sf = {j: int(self.trace["scale_factor"][j]) for j in jobs}
        pw = {j: float(self.pw[j]) for j in jobs}
        since = {j: now - float(self.trace["arrival"][j]) for j in jobs}
        remaining = {j: int(st["total_steps"][s, j] - steps_run[s, j]) for j in jobs}
        name = pol.name
        if name == "AlloX_Perf":
            a = pol.get_allocation(thr, sf, since, remaining, [dict(r) for r in self.per_round_schedule[s]], self.cluster_spec)
        elif name.startswith("FinishTimeFairness"):
            a = pol.get_allocation(thr, sf, pw, since, remaining, self.cluster_spec)
        elif name.startswith("Isolated"):
            a = pol.get_allocation(thr, sf, self.cluster_spec)
        elif name.startswith("MaxMinFairness"):
            a = pol.get_allocation(thr, sf, pw, self.cluster_spec)
        elif name.startswith("MinTotalDuration"):
            a = pol.get_allocation(thr, sf, remaining, self.cluster_spec)
        else:
            a = pol.get_allocation(thr, sf, self.cluster_spec)
        out = np.full((self.J, self.W), np.nan)
        for j, row in (a or {}).items():
            for i, w in enumerate(self.types):
                out[j, i] = row[w]
        self.allocations[s] += 1
        return out

    def run(self, max_rounds=None):
        sim, S, J, G, W, half = self.sim, self.S, self.J, self.ngpus, self.W, self.tpi / 2.0
        scn = sim.begin()
        status = sim.status.copy()
        live_prev = np.zeros((S, J), bool)
        job_time = np.zeros((S, J, W)); deficit = np.zeros((S, J, W)); alloc = np.full((S, J, W), np.nan)
        worker_time = np.zeros((S, W)); last_reset = np.zeros(S); need_update = np.zeros(S, bool)
        prev = [dict() for _ in range(S)]                  # job -> worker ids of the round before (lease extension)
        wtime = np.zeros((S, G))                           # _cumulative_worker_time_so_far
        lease_ext = np.zeros(S, np.int64); lease_opp = np.zeros(S, np.int64)
        sf_all = np.asarray(self.trace["scale_factor"], dtype=np.int32)
        # worker ids are handed out type by type in sorted type order (scheduler.py:1826-1832)
        first = np.concatenate([[0], np.cumsum(self.cap)])
        ids_of = [list(range(int(first[i]), int(first[i + 1]))) for i in range(W)]
        type_of_worker = np.repeat(np.arange(W), self.cap)
        base_order = [self.types.index(w) for w in self.ROUND_ORDER if w in self.types] + \
                     [i for i, w in enumerate(self.types) if w not in self.ROUND_ORDER]
        st = sim.job_state()
        steps_run = np.zeros((S, J), np.int64)
        c = 0
        while not scn["done"].all():
            chosen = np.zeros((S, J), np.uint8)
            active = [s for s in range(S) if not scn["done"][s]]
            for s in active:
                now = float(scn["now"][s])
                live = status[s] == 1
                if c > 0 and (live_prev[s] & ~live).any():
                    need_update[s] = True                                      # _remove_job :903
                new = live & ~live_prev[s]
                if new.any():                                                   # add_job :738-744
                    job_time[s, new] = half
                    deficit[s, new] = 0.0
                    alloc[s, new] = np.nan
                    need_update[s] = True
                live_prev[s] = live
                # _update_priorities :3611-3636
                since = now - last_reset[s]
                if need_update[s] and (since >= self.min_reset or last_reset[s] == 0):
                    jobs = np.flatnonzero(live)
                    for w in range(W):                                          # _reset_time_run_so_far :3498-3551
                        wsum = 0.0
                        for j in jobs.tolist():
                            received = job_time[s, j, w] - half
                            should = 0 if np.isnan(alloc[s, j, w]) else alloc[s, j, w] * since
                            deficit[s, j, w] += should - received
                            job_time[s, j, w] = half
                            wsum += half
                        worker_time[s, w] = wsum
                    last_reset[s] = now
                    alloc[s] = self._allocation(s, live, now, st, steps_run)
                    need_update[s] = False
                jobs = np.flatnonzero(live)
                loc = {int(j): i for i, j in enumerate(jobs.tolist())}
                pv = {loc[j]: (int(type_of_worker[w[0]]), tuple(w)) for j, w in prev[s].items() if j in loc}
                name = self.policies[s].name
                order = list(base_order)
                if "Perf" not in name and "Packing" not in name and W > 1:
                    names = [self.types[i] for i in order]
                    self._shufflers[s].shuffle(names)                          # scheduler.py:1297-1301
                    order = [self.types.index(w) for w in names]
                thr = self.thr_w[jobs] if self.thr_w is not None else st["throughput"][s, jobs][:, None]
                prio, sel, asg = self.backend.gavel_round(
                    alloc[s, jobs], job_time[s, jobs], worker_time[s].copy(), thr, deficit[s, jobs], sf_all[jobs],
                    self.cap.copy(), order, [ids_of[i] for i in order], pv,
                    isolated_plus=(name == "Isolated_plus"), fifo=name.startswith("FIFO"))
                rnd = {int(jobs[i]): tuple(int(w) for w in ws) for i, ws in asg}
                ids = list(rnd)                  # a selected job the allocation does not know yet gets no workers (:1363-1366)
                lease_opp[s] += sum(1 for j in prev[s] if live[j])              # scheduler.py:2198-2213
                lease_ext[s] += sum(1 for j, ws in rnd.items() if j in prev[s] and set(prev[s][j]) == set(ws))
                prev[s] = rnd
                for j in ids:
                    chosen[s, j] = 1 + int(type_of_worker[rnd[j][0]])
                self.per_round_schedule[s].append({j: rnd[j] for j in ids})
            scn = sim.step(chosen)
            if (scn["err"] != 0).any():
                raise RuntimeError(f"swb_sim_step: error flags {scn['err'].tolist()}")
            status = sim.status.copy()
            st = sim.job_state()
            steps_run = sim.results()["steps_run"]
            for s in active:                                                    # the round's completion callbacks
                ran = np.flatnonzero(st["ran"][s])
                for j in sorted(ran.tolist(), key=lambda j: (-st["finish_time"][s, j], j)):
                    if st["failed_attempts"][s, j] > 0:
                        need_update[s] = True                                  # scheduler.py:4569
                    else:
                        ex = float(st["exec_time"][s, j])                      # :4660-4676
                        w = int(chosen[s, j]) - 1
                        job_time[s, j, w] += ex
                        worker_time[s, w] += ex
                        for wid in prev[s].get(j, ()):
                            wtime[s, wid] += ex
            c += 1
            if max_rounds is not None and c >= max_rounds:
                break
        res = sim.results()
        res.update(makespan=scn["now"].copy(), rounds=scn["rounds"].copy(), per_round_schedule=self.per_round_schedule,
                   allocations=self.allocations.copy(), avg_jct=np.nanmean(res["jct"], axis=1),
                   worker_time=wtime, num_lease_extensions=lease_ext, num_lease_extension_opportunities=lease_opp)
        self.last = res
        return res

    def result_dicts(self, isolated_durations, res=None, trace_file=None):
        """One dict per scenario with the keys of the reference's result pickle
        (scripts/drivers/simulate_scheduler_with_trace.py:128-151) — here WITH the worker-dependent ones: per-worker
        utilisation (scheduler.py:3037-3058), lease-extension counts (:2198-2213, :3086-3107), `{job: worker ids}` per
        round.  isolated_durations[j] = sum(profile["duration_every_epoch"]) (finish-time fairness, :2865-2925).
        Absent: envy lists, the Themis variant of the fairness list, the throughput timeline."""
        res = self.last if res is None else res
        J, G = self.J, self.ngpus
        contention = max(1.0, J / G)
        out = []
        for s in range(self.S):
            jct = res["jct"][s]
            done = np.isfinite(jct)
            jl = [float(v) for v in jct[done]]
            util = [round(float(t) / float(res["makespan"][s]), 5) for t in res["worker_time"][s]]
            opp = int(res["num_lease_extension_opportunities"][s])
            ext = int(res["num_lease_extensions"][s])
            out.append({
                "trace_file": trace_file, "policy": self.policies[s].name, "scenario": s,
                "makespan": float(res["makespan"][s]), "avg_jct": float(np.mean(jl)) if jl else None,
                "geometric_mean_jct": float(np.exp(np.mean(np.log(jl)))) if jl else None,
                "harmonic_mean_jct": float(len(jl) / np.sum(1.0 / np.asarray(jl))) if jl else None,
                "jct_list": jl,
                "finish_time_fairness_list": [round(float(jct[j]) / (float(isolated_durations[j]) * contention), 5)
                                              for j in range(J) if done[j]],
                "cluster_util": float(np.mean(util)), "utilization_list": util,
                "extension_percentage": (100.0 * ext) / opp if opp > 0 else 0,
                "num_lease_extensions": ext, "num_lease_extension_opportunities": opp,
                "per_round_schedule": res["per_round_schedule"][s],
                "job_run_time": {j: float(res["run_time"][s, j]) for j in range(J)},
                "time_per_iteration": self.tpi})
        return out
