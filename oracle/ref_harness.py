"""CPU ORACLE tooling (test infrastructure): run the UNMODIFIED reference simulator here.

`/root/reference/scheduler/scheduler.py` (the round mechanism + simulator, SURVEY.md §2 "caller")
cannot be imported as-is in this container: cvxpy / gurobipy / mosek / matrix_completion and the
generated gRPC stubs are absent.  This module
  1. copies the reference's `scheduler/` python files + the canonical trace into a scratch dir
     (the reference writes next to its sources: scheduler.py:126-133, utils.py:1432-1437),
  2. puts empty stand-in modules for the missing third-party names on `sys.modules`,
  3. substitutes the module `shockwave` (the Gurobi-backed solver) by a module holding a
     caller-supplied `ShockwaveScheduler` class — the drop-in boundary of SURVEY.md §8(b),
  4. runs `Scheduler.simulate()` exactly like `scripts/drivers/simulate_scheduler_with_trace.py:21-165`
     and returns the same result dictionary that script pickles.

Nothing here is imported by the product; it exists to (a) pin the oracle against the reference's
golden pickles and (b) record solver-input fixtures for the GPU parity tests.  It works where the reference's
scheduler/ directory exists or where build() made its byte-compiled copy under oracle/_ref (see oracle/stage_ref.py).
"""
from __future__ import annotations

import importlib
import json
import os
import shutil
import sys
import tempfile
import types

_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _find_ref():
    """The reference's scheduler/ directory: $SWB_REF_SCHEDULER, else /root/reference (build container), else the
    byte-compiled build under oracle/_ref (git-ignored, made by build(); see oracle/stage_ref.py)."""
    for cand in (os.environ.get("SWB_REF_SCHEDULER"), "/root/reference/scheduler",
                 os.path.join(_ROOT, "oracle", "_ref", "scheduler")):
        if cand and os.path.isdir(cand):
            return cand
    return "/root/reference/scheduler"


REF = _find_ref()
GOLDEN_DIR = os.path.join(REF, "reproduce", "pickles", "tacc_32gpus")
CANONICAL_TRACE = "traces/reproduce/120_0.2_5_100_40_25_0,0.5,0.5_0.6,0.3,0.09,0.01_multigpu_dynamic.trace"

_STUB_NAMES = [
    "gurobipy", "mosek", "matrix_completion",
    "worker_to_scheduler_pb2", "worker_to_scheduler_pb2_grpc",
    "iterator_to_scheduler_pb2", "iterator_to_scheduler_pb2_grpc",
    "scheduler_to_worker_pb2", "scheduler_to_worker_pb2_grpc", "common_pb2",
    "enums_pb2",
]


def reference_available():
    return os.path.isdir(REF)


def _install_stubs():
    class _Any(types.ModuleType):
        def __getattr__(self, name):
            if name.startswith("__"):
                raise AttributeError(name)
            return type(name, (), {})
    for name in _STUB_NAMES:
        if name not in sys.modules:
            sys.modules[name] = _Any(name)
    if "cvxpy" not in sys.modules:
        cp = _Any("cvxpy")
        cp.__path__ = []
        for sub in ["cvxpy.constraints", "cvxpy.constraints.nonpos", "cvxpy.reductions",
                    "cvxpy.reductions.solvers", "cvxpy.reductions.solvers.defines", "cvxpy.error"]:
            m = _Any(sub)
            m.__path__ = []
            sys.modules[sub] = m
        sys.modules["cvxpy.reductions.solvers.defines"].SOLVER_MAP_CONIC = {}
        sys.modules["cvxpy.error"].DCPError = type("DCPError", (Exception,), {})
        sys.modules["cvxpy"] = cp


def prepare_tree(scratch=None, trace=CANONICAL_TRACE):
    """Copy the reference python tree (no 68 MB traces dir) into a writable scratch dir."""
    scratch = scratch or tempfile.mkdtemp(prefix="swref_")
    dst = os.path.join(scratch, "repo", "scheduler")
    if not os.path.isdir(dst):
        shutil.copytree(REF, dst, ignore=shutil.ignore_patterns("traces", "reproduce", "scripts", "*.png", "__pycache__"))
        os.makedirs(os.path.join(dst, os.path.dirname(trace)), exist_ok=True)
        shutil.copy(os.path.join(REF, trace), os.path.join(dst, trace))
    return dst


def import_reference(dst, shockwave_scheduler_cls=None):
    """Import the copied reference `scheduler` + `utils` modules with stand-ins in place."""
    _install_stubs()
    # scheduler/ first (so `shockwave` is scheduler/shockwave.py, not policies/shockwave.py);
    # the reference itself only *appends* policies/ (policies/policy.py:3).
    if dst not in sys.path:
        sys.path.insert(0, dst)
    for p in (os.path.join(dst, "policies"), os.path.join(dst, "runtime", "rpc")):
        if p not in sys.path:
            sys.path.append(p)
    if shockwave_scheduler_cls is not None:
        mod = types.ModuleType("shockwave")
        mod.ShockwaveScheduler = shockwave_scheduler_cls
        sys.modules["shockwave"] = mod
    else:
        sys.modules.pop("shockwave", None)
    for name in ("scheduler", "utils"):
        sys.modules.pop(name, None)
    ref_utils = importlib.import_module("utils")
    ref_sched = importlib.import_module("scheduler")
    return ref_sched, ref_utils


def simulate(policy_name, shockwave_scheduler_cls=None, policy_obj=None,
             config="configurations/tacc_32gpus.json", cluster="32:0:0", trace=CANONICAL_TRACE,
             throughputs="tacc_throughputs.json", time_per_iteration=120, seed=0, scratch=None,
             max_rounds=None, scheduler_mixin=None, extract=None):
    """Mirror of simulate_scheduler_with_trace.py:main for one policy.  Returns the result dict (+ `extra` =
    extract(scheduler, jobs, arrival_times) when a callback is given: internal records for the simulator pins)."""
    dst = prepare_tree(scratch, trace)
    cwd = os.getcwd()
    os.chdir(dst)
    try:
        ref_sched, ref_utils = import_reference(dst, shockwave_scheduler_cls)
        import pickle
        trace_file = os.path.join(dst, trace)
        throughputs_file = os.path.join(dst, throughputs)
        jobs, arrival_times = ref_utils.generate_pickle_file(trace_file, throughputs_file)
        if policy_obj is None:
            policy_obj = ref_utils.get_policy(policy_name, solver="ECOS", seed=seed)
        pickle_path = os.path.splitext(trace_file)[0] + ".pickle"
        with open(pickle_path, "rb") as f:
            tp = pickle.load(f)
        for job_id, job in enumerate(jobs):
            job.duration = sum(tp[job_id]["duration_every_epoch"])
        n = [int(v) for v in cluster.split(":")]
        cluster_spec = {"v100": n[0], "p100": n[1], "k80": n[2]}
        per_server = {"v100": 1, "p100": 1, "k80": 1}
        sw_cfg = None
        if policy_name == "shockwave":
            sw_cfg = json.load(open(os.path.join(dst, config)))
            sw_cfg["time_per_iteration"] = time_per_iteration
            sw_cfg["num_gpus"] = cluster_spec["v100"] * per_server["v100"]
        sched_cls = ref_sched.Scheduler
        if scheduler_mixin is not None:      # drop-in for methods of the round mechanism itself (placement.py)
            sched_cls = type("Scheduler", (scheduler_mixin, ref_sched.Scheduler), {})
        sched = sched_cls(policy_obj, throughputs_file=throughputs_file, simulate=True,
                                    seed=seed, time_per_iteration=time_per_iteration,
                                    pickle_file=pickle_path, shockwave_config=sw_cfg)
        makespan = sched.simulate(cluster_spec, arrival_times, jobs,
                                  num_gpus_per_server=per_server, jobs_to_complete=None)
        avg_jct, _, _, jct_list = sched.get_average_jct(job_ids=None)
        util, _ = sched.get_cluster_utilization()
        ftf_list, _ = sched.get_finish_time_fairness(job_ids=None,
                                                     pickle_file_name=f"{trace_file}.pickle")
        out = dict(makespan=makespan, avg_jct=avg_jct, jct_list=jct_list, cluster_util=util,
                   finish_time_fairness_list=ftf_list,
                   per_round_schedule=sched.get_per_round_schedule())
        if extract is not None:
            out["extra"] = extract(sched, jobs, arrival_times)
        sched.shutdown()
        return out
    finally:
        os.chdir(cwd)


# ---------------------------------------------------------------------------------------------
# Oracle-backed ShockwaveScheduler: the product's host state machine with the device calls replaced
# by (a) the REFERENCE's own JobMetaData methods for the forecast and (b) oracle/shockwave_milp.py
# (HiGHS) for the solve.  Used to pin the oracle against the golden pickles and to record fixtures.
# ---------------------------------------------------------------------------------------------
def make_oracle_scheduler_cls(record=None, rel_gap=1e-3, time_limit=15.0, placement=None, key_stats=None):
    """placement: optional callable(n, g, G, T, bfkey, fallback=, w=) -> dict(x=...) that replaces the solver's own x
    (and the re-rank MILP) by a placement RULE applied to the solver's round counts — used to run the product's placement
    rule (tests/ref_placement.py, the numpy restatement of place.cu) closed-loop.
    key_stats: optional dict; filled with how often the reference's PER-ROUND back-fill sort keys (one
    dirichlet_posterior_remaining_runtime() call per idle round and unscheduled job, each of which recalibrates:
    shockwave.py:261-267 -> JobMetaData.py:355 -> :302) differ from the job's FIRST key of the same re-solve, and how many
    rounds would be back-filled differently with first keys only (what place.cu sorts on, DESIGN.md section 3)."""
    import random as _random

    import numpy as _np

    from oracle import shockwave_milp as om
    from shockwave_b200.scheduler import ShockwaveScheduler as _Base

    statics = {}

    class OracleShockwaveScheduler(_Base):
        job_statics = statics

        def _on_add(self, jobid, job):
            pass

        def _on_remove(self, jobid):
            pass

        def _resolve(self, jobids, jobobjs):
            J = len(jobids)
            G, T, D, r = self.ngpus, self.future_nrounds, self.round_duration, self.round_ptr
            tl = [self._timeline_summary(jid, job) for jid, job in zip(jobids, jobobjs)]
            reest = bool(self.reestimate_share)
            if record is not None:
                for jid, job in zip(jobids, jobobjs):
                    if jid not in statics:
                        statics[jid] = dict(nworkers=job.nworkers, epochs=job.epochs,
                                            epoch_nsamples=job.epoch_nsamples,
                                            timestamp_submit=job.timestamp_submit,
                                            pre=_np.asarray(job.epoch_duration_preprofiled, dtype=_np.float64),
                                            bs=_np.asarray(job.bs_schedule, dtype=_np.int32),
                                            grd=job.gavel_round_duration)
            # finish_time_uniform_share, shockwave.py:88-120 (reference objects, reference call order)
            if self.reestimate_share:
                for jobid, job in zip(jobids, jobobjs):
                    share = min(1.0, G / J)
                    job.calibrate_profiled_epoch_duration()
                    est = job.timestamp_submit + (
                        sum(job.epoch_duration[: job.epoch_progress])
                        + job.dirichlet_posterior_remaining_runtime(job.epoch_progress)) / share
                    self.share_series.setdefault(jobid, []).append((r, est))
            dbar = _np.empty(J); R = _np.empty(J); ftobj = _np.empty(J)
            for i, job in enumerate(jobobjs):                      # shockwave.py:322-324
                job.calibrate_profiled_epoch_duration()
                dbar[i] = _np.mean(job.epoch_duration[: job.epoch_progress + 1])
            for i, job in enumerate(jobobjs):                      # shockwave.py:558-562
                R[i] = job.dirichlet_posterior_remaining_runtime()
            for i, jobid in enumerate(jobids):                     # shockwave.py:588-590
                ftobj[i] = om.finish_time_momentumed_average(list(self.share_series[jobid]), r)
            g = _np.array([job.nworkers for job in jobobjs], dtype=_np.int64)
            E = _np.array([job.epochs for job in jobobjs], dtype=_np.int64)
            c = _np.array([job.epoch_progress for job in jobobjs], dtype=_np.int64)
            logv = om.pwl_log_values(self.logapx_bases, self.logapx_origin)
            _random.seed(0); _np.random.seed(0)                    # shockwave.py:451-452
            ones = _np.ones(J)
            cap = om.ftf_caps(R, ftobj, G, J, T, D, r, self.rhomax)
            ok, x, p, obj = om._solve(g, E.astype(float), c.astype(float), dbar, R, ones, G, T, D, self.k,
                                      self.logapx_bases, logv, cap, rel_gap, time_limit)
            status, weights, R_fb = om.STATUS_FTF_FEASIBLE, ones, None
            if not ok:
                status = om.STATUS_FALLBACK
                R_fb = _np.empty(J)
                for i, job in enumerate(jobobjs):                  # shockwave.py:863-866
                    job.calibrate_profiled_epoch_duration()
                    R_fb[i] = job.dirichlet_posterior_remaining_runtime()
                weights, _ = om.relax_priorities(R_fb, ftobj, G, J, D, r, self.rhomax, self.lam)
                ok, x, p, obj = om._solve(g, E.astype(float), c.astype(float), dbar, R, weights, G, T, D,
                                          self.k, self.logapx_bases, logv, None, rel_gap, time_limit)
                assert ok
                if placement is None:
                    x = om.rank_in_schedule(x, weights, g, G, rel_gap, time_limit)
            if placement is not None:
                counts = _np.round(_np.asarray(x)).sum(axis=1).astype(_np.int64)
                placed = placement(counts, g, G, T, _np.zeros(J), fallback=(status == om.STATUS_FALLBACK), w=weights)
                assert placed["shortfall"] == 0, "the placement rule could not seat the solver's counts"
                x = placed["x"].astype(float)
            # construct_schedules, shockwave.py:213-285, with the reference's per-round sort-key calls
            sched = OrderedDict()
            bfkey0 = _np.full(J, _np.nan)
            for t in range(T):
                cur = [i for i in range(J) if round(float(x[i, t])) == 1.0]
                idle = G - int(sum(g[i] for i in cur))
                names = [jobids[i] for i in cur]
                if idle > 0:
                    non = [i for i in range(J) if i not in set(cur)]
                    keys = {i: jobobjs[i].dirichlet_posterior_remaining_runtime() for i in non}
                    if t == 0:
                        for i, v in keys.items():
                            bfkey0[i] = v
                    if key_stats is not None:
                        first = key_stats.setdefault("_first", {})
                        for i, v in keys.items():
                            first.setdefault((r, jobids[i]), v)
                        k0 = {i: first[(r, jobids[i])] for i in non}
                        key_stats["keys"] = key_stats.get("keys", 0) + len(keys)
                        key_stats["keys_differ"] = key_stats.get("keys_differ", 0) + sum(1 for i in non if keys[i] != k0[i])
                        key_stats["idle_rounds"] = key_stats.get("idle_rounds", 0) + 1
                        a = sorted(non, key=lambda i: keys[i], reverse=True)
                        b = sorted(non, key=lambda i: k0[i], reverse=True)
                        def fill(order, idle=idle):
                            got = []
                            for i in order:
                                if g[i] <= idle:
                                    idle -= int(g[i]); got.append(i)
                                if idle <= 0:
                                    break
                            return got
                        key_stats["rounds_filled_differently"] = key_stats.get("rounds_filled_differently", 0) + (fill(a) != fill(b))
                        key_stats["first_rounds_filled_differently"] = key_stats.get("first_rounds_filled_differently", 0) + (
                            t == 0 and fill(a) != fill(b))
                    for i in sorted(non, key=lambda i: keys[i], reverse=True):
                        if g[i] <= idle:
                            idle -= int(g[i])
                            names.append(jobids[i])
                        if idle <= 0:
                            break
                sched[r + t] = names
            ev = om.evaluate(x, g, E.astype(float), c.astype(float), dbar, R, weights, G, T, D, self.k,
                             self.logapx_bases, logv)
            self.last_result = dict(status=status, objective=ev[0], welfare=ev[1], makespan=ev[2])
            if record is not None:
                record.append(dict(round_ptr=r, J=J, g=g.copy(), E=E.copy(), c=c.copy(), dbar=dbar.copy(),
                                   rem=R.copy(), ftobj=ftobj.copy(), rem_fb=None if R_fb is None else R_fb.copy(),
                                   bfkey0=bfkey0, status=status, objective=ev[0], welfare=ev[1],
                                   makespan=ev[2], x=x.astype(_np.uint8), weights=_np.asarray(weights).copy(),
                                   jobids=list(jobids), round0=list(sched[r]),
                                   reestimate=reest, meas_ns=_np.array([t[0] for t in tl]),
                                   meas_end=_np.array([t[1] for t in tl], dtype=_np.int32)))
            return sched

    from collections import OrderedDict
    return OracleShockwaveScheduler
