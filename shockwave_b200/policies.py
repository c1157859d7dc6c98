"""Gavel policies behind the reference's own `get_allocation()` signatures, solved on the GPU.

Mirrors scheduler/policies/{policy,max_min_fairness,finish_time_fairness,min_total_duration,
max_sum_throughput,isolated,proportional,gandiva_fair_proportional}.py: same class names, same `.name`
strings (scheduler.py:3291-3355 dispatches on their prefixes), same positional arguments, same
`{job_id: {worker_type: fraction}}` return value and `None` for an empty job set (policy.py:31-32).

The LP each policy hands to cvxpy is solved on the GPU (no CPU fallback):
  * swb_policy_pooled (policy.cu) when all worker types WITH capacity give a job the same throughput — always
    true for the non-Perf classes (they overwrite the matrix with the v100 column, or with 1.0) and for the
    homogeneous clusters Shockwave targets: closed forms / 1-D searches;
  * swb_policy_hetero (hetero.cu) for genuinely heterogeneous *_Perf calls with up to 3 worker types that have
    capacity (k80 / p100 / v100): bisection on the scalar objective + Dantzig-Wolfe on the capacity rows.
More than 4 live worker types (3 for max-sum; e.g. all six of tacc_throughputs.json) go to swb_lp_solve as general
LPs (packing.hetero_lp; up to ~1000 jobs), and so do the *_packed policies (packing.py).
"""
from __future__ import annotations

import copy
import ctypes as C
import operator
import os

import numpy as np

from . import engine as _eng

POL_MAXMIN, POL_FTF, POL_MTD, POL_MAXSUM, POL_ISOLATED = 1, 2, 3, 4, 5

_shared_engine = None
_device = int(os.environ.get("SWB_DEVICE", "0"))


def set_device(device):
    """CUDA device the policy kernels run on (default: $SWB_DEVICE or 0).  Drops the engine of another device."""
    global _shared_engine, _device
    if int(device) != _device and _shared_engine is not None:
        _shared_engine.close()
        _shared_engine = None
    _device = int(device)


def _engine():
    global _shared_engine
    if _shared_engine is None:
        _shared_engine = _eng.Engine(_device)
    return _shared_engine


def _pooled(mode, N, coef, sf, t=None, n=None, den=None):
    eng = _engine()
    lib = eng.lib
    arr = lambda a: None if a is None else np.ascontiguousarray(a, dtype=np.float64)
    coef, sf, t, n, den = arr(coef), arr(sf), arr(t), arr(n), arr(den)
    J = len(coef)
    x = np.zeros(J, dtype=np.float64)
    obj = C.c_double()
    p = lambda a: None if a is None else C.c_void_p(a.ctypes.data)
    rc = lib.swb_policy_pooled(eng.h, mode, J, float(N), p(coef), p(sf), p(t), p(n), p(den), p(x), C.byref(obj))
    if rc < 0:
        raise RuntimeError(f"swb_policy_pooled failed ({rc}): {lib.swb_last_error().decode()}")
    return x, obj.value, rc


def _hetero(mode, N, a, sf, t=None, n=None, den=None):
    """swb_policy_hetero on the live worker types: a is J x W, N has W entries > 0.  Returns (x[J,W], objective, rc)."""
    W_ = np.shape(a)[1]
    if W_ > 4 or (mode == POL_MAXSUM and W_ > 3):
        # beyond the basis enumeration of hetero.cu's master: the same program as a general LP on swb_lp_solve
        from . import packing
        out = packing.hetero_lp(mode, N, a, sf, t=t, n=n, den=den)
        _hetero.last_stats = (0, 0)
        return out
    eng = _engine()
    lib = eng.lib
    arr = lambda v: None if v is None else np.ascontiguousarray(v, dtype=np.float64)
    a, sf, t, n, den, N = arr(a), arr(sf), arr(t), arr(n), arr(den), arr(N)
    J, W = a.shape
    x = np.zeros((J, W), dtype=np.float64)
    obj = C.c_double()
    stats = np.zeros(2, dtype=np.int32)
    p = lambda v: None if v is None else C.c_void_p(v.ctypes.data)
    rc = lib.swb_policy_hetero(eng.h, mode, J, W, p(N), p(a), p(sf), p(t), p(n), p(den), p(x), C.byref(obj),
                               p(stats))
    if rc < 0:
        raise RuntimeError(f"swb_policy_hetero failed ({rc}): {lib.swb_last_error().decode()}")
    _hetero.last_stats = (int(stats[0]), int(stats[1]))
    return x, obj.value, rc


class Policy:
    """policy.py:11-65."""
    def __init__(self, solver="ECOS"):
        self._name = None
        self._solver = solver       # kept for signature parity; no CPU solver is ever called

    @property
    def name(self):
        return self._name

    def flatten(self, d, cluster_spec):
        job_ids = sorted(list(d.keys()))
        if len(job_ids) == 0:
            return None, None
        worker_types = sorted(list(d[job_ids[0]].keys()))
        self._num_workers = [cluster_spec[w] for w in worker_types]
        if len(worker_types) == 0:
            return None, None
        # the dict-of-dicts walk runs in C: map + itemgetter instead of a nested Python loop
        rows = map(d.__getitem__, job_ids)
        if len(worker_types) == 1:
            m = np.fromiter(map(operator.itemgetter(worker_types[0]), rows), dtype=np.float64,
                            count=len(job_ids)).reshape(-1, 1)
        else:
            m = np.array(list(map(operator.itemgetter(*worker_types), rows)), dtype=np.float64)
        return m, (job_ids, worker_types)

    def unflatten(self, m, index):
        job_ids, worker_types = index
        return {jid: dict(zip(worker_types, row)) for jid, row in zip(job_ids, np.asarray(m).tolist())}

    # ---- pooling of the worker types (see module docstring) ----
    def _pool(self, throughputs):
        N = np.asarray(self._num_workers, dtype=np.float64)
        live = N > 0
        if not live.any():
            raise ValueError("cluster has no workers")
        cols = throughputs[:, live]
        if not np.allclose(cols, cols[:, :1], rtol=1e-12, atol=0.0):
            return None, float(N.sum()), N / N.sum()       # heterogeneous: the caller goes through _solve_hetero
        return cols[:, 0].copy(), float(N.sum()), N / N.sum()

    def _solve_hetero(self, mode, a, sf, t=None, n=None, den=None):
        """a: J x W matrix over ALL worker types; types without capacity get x = 0."""
        N = np.asarray(self._num_workers, dtype=np.float64)
        live = N > 0
        x_live, obj, rc = _hetero(mode, N[live], a[:, live], sf, t=t, n=n, den=den)
        x = np.zeros_like(a, dtype=np.float64)
        x[:, live] = x_live
        return np.clip(x, 0.0, 1.0), obj, rc

    @staticmethod
    def _split(x, share):
        return np.clip(x[:, None] * share[None, :], 0.0, 1.0)


class ProportionalPolicy(Policy):
    def __init__(self):
        self._name = "Proportional"

    def get_allocation(self, unflattened_throughputs, cluster_spec):
        throughputs, index = super().flatten(unflattened_throughputs, cluster_spec)
        if throughputs is None:
            return None
        m = throughputs.shape[0]
        N = np.asarray(self._num_workers, dtype=np.float64)
        # proportional.py:36-43: x_jw = N_w/m divided by the (common) row sum -> N_w / sum N; a constant
        # matrix, there is nothing to solve
        return super().unflatten(np.tile(N / N.sum(), (m, 1)) if N.sum() > 0 else np.zeros_like(throughputs), index)


class IsolatedPolicy(Policy):
    def __init__(self):
        self._name = "Isolated"

    def _alloc(self, throughputs, sf):
        N = np.asarray(self._num_workers, dtype=np.float64)
        x, _, _ = _pooled(POL_ISOLATED, N.sum(), sf, sf)     # min(1, (sum N / m) / sf_j)  (isolated.py:46-53)
        share = N / N.sum() if N.sum() > 0 else N
        return x[:, None] * share[None, :]

    def get_allocation(self, unflattened_throughputs, scale_factors, cluster_spec):
        throughputs, index = super().flatten(unflattened_throughputs, cluster_spec)
        if throughputs is None:
            return None
        sf = np.array([scale_factors[j] for j in index[0]], dtype=np.float64)
        return super().unflatten(self._alloc(throughputs, sf), index)


class GandivProportionalPolicy(Policy):
    def __init__(self):
        self._name = "GandivaFairProportional"

    def get_allocation(self, unflattened_throughputs, scale_factors, cluster_spec):
        throughputs, index = super().flatten(unflattened_throughputs, cluster_spec)
        if throughputs is None:
            return None
        m = throughputs.shape[0]
        N = np.asarray(self._num_workers, dtype=np.float64)
        x, _, _ = _pooled(POL_ISOLATED, N.sum(), np.ones(m), np.ones(m))   # gandiva_fair_proportional.py:26-41
        share = N / N.sum() if N.sum() > 0 else N
        return super().unflatten(x[:, None] * share[None, :], index)


class IsolatedPlusPolicy(GandivProportionalPolicy):
    """isolated_plus.py:10-76: the equal split without the scale-factor division — the same closed form as
    gandiva_fair_proportional.py (x_jw = N_w/m, rows normalised to <= 1)."""
    def __init__(self):
        self._name = "Isolated_plus"


class MaxMinFairnessPolicyWithPerf(Policy):
    def __init__(self, solver):
        Policy.__init__(self, solver)
        self._name = "MaxMinFairness_Perf"

    def get_allocation(self, unflattened_throughputs, scale_factors, unflattened_priority_weights, cluster_spec):
        throughputs, index = super().flatten(unflattened_throughputs, cluster_spec)
        if throughputs is None:
            return None
        job_ids, _ = index
        thr, N, share = self._pool(throughputs)
        sf = np.array([scale_factors[j] for j in job_ids], dtype=np.float64)
        pw = np.array([1.0 / unflattened_priority_weights[j] for j in job_ids], dtype=np.float64)
        if thr is None:
            # proportional.py:20-43: x_jw = N_w / sum N for every job -> proportional throughput sum_w thr_jw N_w / sum N
            prop = throughputs @ share
            coef = throughputs * (pw / prop * sf)[:, None]          # max_min_fairness.py:78-101
            x, self.last_objective, _ = self._solve_hetero(POL_MAXMIN, coef, sf)
            return super().unflatten(x, index)
        # proportional throughput of a pooled job is its own throughput (proportional.py:36-43), so the
        # objective coefficient thr*sf*pw/prop (max_min_fairness.py:78-101) collapses to sf*pw
        coef = thr * sf * pw / thr
        x, self.last_objective, _ = _pooled(POL_MAXMIN, N, coef, sf)
        return super().unflatten(self._split(x, share), index)


class MaxMinFairnessPolicy(Policy):
    def __init__(self, solver):
        self._name = "MaxMinFairness"
        self._max_min_fairness_perf_policy = MaxMinFairnessPolicyWithPerf(solver)

    def get_allocation(self, unflattened_throughputs, scale_factors, priority_weights, cluster_spec):
        throughputs, index = super().flatten(unflattened_throughputs, cluster_spec)
        if throughputs is None:
            return None
        ones = {j: {w: 1.0 for w in unflattened_throughputs[j]} for j in unflattened_throughputs}
        return self._max_min_fairness_perf_policy.get_allocation(ones, scale_factors, priority_weights, cluster_spec)


def _waterfill_step(N, thr, sf, prop, lower, mult, M, slack=1.0001):
    """swb_policy_waterfill_step: the LP and the bottleneck program of one water-filling iteration on the device.
    Returns (x[J,W], c, z[J]) or (None, None, None) when the LP has no feasible point."""
    eng = _engine()
    lib = eng.lib
    arr = lambda v: np.ascontiguousarray(v, dtype=np.float64)
    N, thr, sf, prop, lower, mult = arr(N), arr(thr), arr(sf), arr(prop), arr(lower), arr(mult)
    J, W = thr.shape
    if W > 3:
        raise NotImplementedError("water-filling with more than 3 worker types with capacity: not solved on the GPU in this release")
    x = np.zeros((J, W), dtype=np.float64)
    z = np.zeros(J, dtype=np.float64)
    c = C.c_double()
    stats = np.zeros(4, dtype=np.int32)
    p = lambda v: C.c_void_p(v.ctypes.data)
    rc = lib.swb_policy_waterfill_step(eng.h, J, W, p(N), p(thr), p(sf), p(prop), p(lower), p(mult), float(M),
                                       float(slack), p(x), C.byref(c), p(z), p(stats))
    if rc < 0:
        raise RuntimeError(f"swb_policy_waterfill_step failed ({rc}): {lib.swb_last_error().decode()}")
    _waterfill_step.last_stats = tuple(int(v) for v in stats)
    if rc == 1:
        return None, None, None
    return x, c.value, z


class WaterFillingAlgorithm:
    """max_min_fairness_water_filling.py:13-413: the iteration loop and the entity re-weighting stay on the host (dict
    bookkeeping, a handful of iterations); `_get_allocation` (ECOS LP) and `_get_bottleneck_jobs` (GLPK_MI MILP) are
    one device call per iteration (swb_policy_waterfill_step)."""
    SLACK, EPSILON = 1.0001, 1e-5      # water_filling.py:200-203

    def __init__(self, priority_reweighting_policies):
        self._previous_priority_weights = None
        self._priority_reweighting_policies = priority_reweighting_policies

    def _compute_priority_weights(self, entity_weights, priority_weights, entity_to_job_mapping,
                                  final_normalized_effective_throughputs, job_ids):
        # water_filling.py:16-79
        returned_priority_weights = {}
        if self._priority_reweighting_policies is None:
            return priority_weights
        if entity_to_job_mapping is None:
            raise ValueError("entity_to_job_mapping cannot be None when priority_reweighting_policies is not None!")
        final = final_normalized_effective_throughputs
        for entity_id in entity_to_job_mapping:
            pol = self._priority_reweighting_policies[entity_id]
            entity_weight = entity_weights[entity_id]
            jobs = entity_to_job_mapping[entity_id]
            if pol == "fairness":
                total = 0.0
                for job_id in jobs:
                    if job_id not in final:
                        total += float(priority_weights[job_id])
                for job_id in jobs:
                    returned_priority_weights[job_id] = 0.0 if job_id in final else \
                        entity_weight * (float(priority_weights[job_id]) / total)
            elif pol == "fifo":
                jobs.sort()
                done = False
                for job_id in jobs:
                    if job_id in final or done:
                        returned_priority_weights[job_id] = 0.0
                    else:
                        returned_priority_weights[job_id] = entity_weight
                        done = True
            else:
                raise ValueError("Unknown priority reweighting policy!")
        return returned_priority_weights

    def _run_get_allocation_iterations(self, job_ids, thr, sf, N, prop, M, entity_weights,
                                       unflattened_priority_weights, entity_to_job_mapping, verbose=False):
        """water_filling.py:307-413 on arrays (thr: J x W over the LIVE worker types).  Returns x of the last LP."""
        J = len(job_ids)
        final = {}
        so_far = np.zeros(J)
        x = None
        done = False
        self.last_iterations = 0
        while not done:
            pw_d = self._compute_priority_weights(entity_weights, unflattened_priority_weights, entity_to_job_mapping,
                                                  final, job_ids)
            self._previous_priority_weights = copy.copy(pw_d)
            pw = np.array([1.0 / pw_d[j] if pw_d[j] > 0 else 0.0 for j in job_ids])
            is_final = np.fromiter((j in final for j in job_ids), dtype=bool, count=J)
            active = (~is_final) & (pw > 0.0)
            mult = np.where(active, pw * sf, 0.0)
            lower = np.where(is_final, np.array([final.get(j, 0.0) for j in job_ids]), so_far)
            # the packing class (packing.py) substitutes its own step: general LPs over (combination, type) columns
            step = getattr(self, "_waterfill_step", None) or _waterfill_step
            xs, c, z = step(N, thr, sf, prop, lower, mult, M, self.SLACK)
            if xs is None:                       # "x is None" / solver exception: keep the previous iterate, stop
                done = True
                z = np.zeros(J)
            else:
                x = xs
                so_far = so_far + np.where(active, c / np.where(active, mult, 1.0), 0.0)
                # the reference's MILP also bounds every z = 0 job from above by so_far * slack - epsilon, which no
                # point satisfies for so_far < 0.1: GLPK reports infeasible, the except branch returns z = 0 for all
                lim = so_far * self.SLACK - self.EPSILON
                base = np.where(is_final, lower, so_far)
                if np.any(((~active) | (z < 0.5)) & (lim < base)):
                    z = np.zeros(J)
            before = len(final)
            for i in np.flatnonzero(active & (z < 0.5)).tolist():
                final[job_ids[i]] = so_far[i]
            if verbose:
                print("water-filling iteration %d: c = %.6f, %d saturated" % (self.last_iterations, c or 0.0, len(final)))
            if before == len(final):
                done = True
            self.last_iterations += 1
            if len(final) == J:
                done = True
        self.last_so_far = so_far
        return x


class MaxMinFairnessWaterFillingPolicyWithPerf(Policy, WaterFillingAlgorithm):
    """max_min_fairness_water_filling.py:476-576."""
    def __init__(self, priority_reweighting_policies=None):
        WaterFillingAlgorithm.__init__(self, priority_reweighting_policies)
        Policy.__init__(self, solver=None)
        self._name = "MaxMinFairnessWaterFilling_Perf"

    def get_allocation(self, unflattened_throughputs, scale_factors, unflattened_priority_weights, cluster_spec,
                       entity_weights=None, entity_to_job_mapping=None, verbose=False,
                       return_effective_throughputs=False):
        throughputs, index = super().flatten(unflattened_throughputs, cluster_spec)
        if throughputs is None:
            return None
        job_ids, _ = index
        sf = np.array([scale_factors[j] for j in job_ids], dtype=np.float64)
        Nall = np.asarray(self._num_workers, dtype=np.float64)
        share = Nall / Nall.sum()
        prop = throughputs @ share                                    # proportional.py:20-43
        self._M = float(np.max(throughputs / prop[:, None] * sf[:, None]))     # water_filling.py:507-512
        live = Nall > 0
        thr, Npool, _ = self._pool(throughputs)
        if thr is not None:       # every live type gives a job the same throughput: one pooled type, split by capacity
            xs = self._run_get_allocation_iterations(job_ids, thr[:, None], sf, np.array([Npool]), prop, self._M,
                                                     entity_weights, unflattened_priority_weights,
                                                     entity_to_job_mapping, verbose)
            x = self._split(xs[:, 0], share)
        else:
            xs = self._run_get_allocation_iterations(job_ids, throughputs[:, live], sf, Nall[live], prop, self._M,
                                                     entity_weights, unflattened_priority_weights,
                                                     entity_to_job_mapping, verbose)
            x = np.zeros_like(throughputs)
            x[:, live] = xs
        x = np.clip(x, 0.0, 1.0)
        if return_effective_throughputs:
            return (throughputs * x).sum(axis=1) / prop, job_ids
        return super().unflatten(x, index)


class MaxMinFairnessWaterFillingPolicy(Policy, WaterFillingAlgorithm):
    """max_min_fairness_water_filling.py:416-473: the same algorithm with every throughput set to 1.0."""
    def __init__(self, priority_reweighting_policies=None):
        self._name = "MaxMinFairnessWaterFilling"
        self._max_min_fairness_perf_policy = MaxMinFairnessWaterFillingPolicyWithPerf(priority_reweighting_policies)

    def get_allocation(self, unflattened_throughputs, scale_factors, unflattened_priority_weights, cluster_spec,
                       entity_weights=None, entity_to_job_mapping=None, verbose=False,
                       return_effective_throughputs=False):
        throughputs, index = super().flatten(unflattened_throughputs, cluster_spec)
        if throughputs is None:
            return None
        job_ids, worker_types = index
        ones = {j: {w: 1.0 for w in unflattened_throughputs[j]} for j in unflattened_throughputs}
        unflattened_x = self._max_min_fairness_perf_policy.get_allocation(
            ones, scale_factors, unflattened_priority_weights, cluster_spec, entity_weights=entity_weights,
            entity_to_job_mapping=entity_to_job_mapping, verbose=verbose, return_effective_throughputs=False)
        if return_effective_throughputs:
            x = np.array([[unflattened_x[j][w] for w in worker_types] for j in job_ids])
            Nall = np.asarray(self._num_workers, dtype=np.float64)
            prop = throughputs @ (Nall / Nall.sum())
            return (throughputs * x).sum(axis=1) / prop, job_ids
        return unflattened_x


class MaxMinFairnessStrategyProofPolicy(Policy):
    """max_min_fairness_strategy_proof.py:13-44: max-min fairness with every throughput set to 1.0."""
    def __init__(self, solver):
        self._name = "MaxMinFairness"
        self._max_min_fairness_perf_policy = MaxMinFairnessPolicyWithPerf(solver)

    def get_allocation(self, unflattened_throughputs, scale_factors, priority_weights, cluster_spec):
        throughputs, index = super().flatten(unflattened_throughputs, cluster_spec)
        if throughputs is None:
            return None
        ones = {j: {w: 1.0 for w in unflattened_throughputs[j]} for j in unflattened_throughputs}
        return self._max_min_fairness_perf_policy.get_allocation(ones, scale_factors, priority_weights, cluster_spec)


def _eisenberg_gale(N, coef, sf, present, iters=4000):
    """S Eisenberg-Gale programs in one batch on the device:  max sum_{j present in s} log(sum_w coef_jw x_jw)
    s.t. x >= 0, sum_w x_jw <= 1, sum_j sf_j x_jw <= N_w — the cvxpy geo_mean program of
    max_min_fairness_strategy_proof.py:102-123.  present [S][J] bool.  Solved by the dense price-response kernel
    (market.cu, log utility) on a 4-round tensor with constant capacities; returns x [S][J][W].  4000 passes: the
    iteration converges linearly once the active set is found, which takes a few hundred to ~2500 passes on the test
    instances (numpy restatement: utilities within 1e-5 of the oracle's after 3000)."""
    S, J = present.shape
    W, T = len(N), 4
    eng = _engine()
    prm = [_eng.make_params(int(max(1, round(float(np.sum(N))))), T, 1.0, 0.0, 1.0, 1.0, [0.0, 1.0], {0.0: 1e-6})] * S
    rate = np.ascontiguousarray(np.broadcast_to((coef / T)[None], (S, J, W)), dtype=np.float32)
    g = np.ascontiguousarray(np.broadcast_to(np.asarray(sf, np.int32)[None], (S, J)))
    E = np.ascontiguousarray(present, dtype=np.float64)
    zeros, ones = np.zeros((S, J)), np.ones((S, J))
    X = np.zeros((S, J, W, T), dtype=np.float32)
    _eng.market_pgd(eng, prm, g, E, zeros, ones, zeros, rate, np.asarray(N, np.float64), X, iters, utility=1)
    return X.mean(axis=3, dtype=np.float64) * present[:, :, None]


class MaxMinFairnessStrategyProofPolicyWithPerf(Policy):
    """max_min_fairness_strategy_proof.py:47-155: the Nash-welfare (geo_mean) allocation, discounted per job by the
    product over the OTHER jobs of (their throughput with the job) / (their throughput without it) — J + 1
    Eisenberg-Gale programs, solved here as ONE batch of J + 1 scenarios by the dense price-response kernel."""
    def __init__(self, solver):
        Policy.__init__(self, solver)
        self._name = "MaxMinFairness_Perf"

    def get_allocation(self, unflattened_throughputs, scale_factors, unflattened_priority_weights, cluster_spec,
                       recurse_deeper=True):
        throughputs, index = super().flatten(unflattened_throughputs, cluster_spec)
        if throughputs is None:
            return None
        m, n = throughputs.shape
        job_ids, _ = index
        N = np.asarray(self._num_workers, dtype=np.float64)
        live = N > 0
        if not live.any():
            raise ValueError("cluster has no workers")
        sf = np.array([scale_factors[j] for j in job_ids], dtype=np.float64)
        pw = np.array([1.0 / unflattened_priority_weights[j] for j in job_ids], dtype=np.float64)
        prop = throughputs @ (N / N.sum())                          # proportional.py:20-43
        coef = throughputs * (pw / prop * sf)[:, None]              # :87-116
        present = np.ones((m + 1 if recurse_deeper else 1, m), dtype=bool)
        for i in range(m if recurse_deeper else 0):
            present[i + 1, i] = False                               # scenario i + 1: the market without job i (:68-84)
        x_live = _eisenberg_gale(N[live], coef[:, live], sf, present)
        x = np.zeros((present.shape[0], m, n))
        x[:, :, live] = x_live
        thr = (throughputs[None] * x).sum(axis=2)                   # :130-133, per scenario
        if not recurse_deeper:
            return {job_ids[i]: thr[0, i] for i in range(m)}
        discount = np.ones(m)
        for i in range(m):                                          # :137-145
            others = present[i + 1]
            discount[i] = float(np.prod(thr[0, others] / thr[i + 1, others])) if others.any() else 1.0
        alloc = (x[0].T * discount).T
        return super().unflatten(alloc.clip(min=0.0).clip(max=1.0), index), discount


class FinishTimeFairnessPolicyWithPerf(Policy):
    def __init__(self, solver):
        Policy.__init__(self, solver)
        self._name = "FinishTimeFairness_Perf"
        self._isolated_policy = IsolatedPolicy()
        self._cumulative_isolated_time = {}
        self._isolated_throughputs_prev_iteration = {}
        self._num_steps_remaining_prev_iteration = {}

    def get_allocation(self, unflattened_throughputs, scale_factors, unflattened_priority_weights,
                       times_since_start, num_steps_remaining, cluster_spec):
        throughputs, index = super().flatten(unflattened_throughputs, cluster_spec)
        if throughputs is None:
            self._isolated_throughputs_prev_iteration = {}
            self._num_steps_remaining_prev_iteration = {}
            return None
        job_ids, _ = index
        thr, N, share = self._pool(throughputs)
        sf = np.array([scale_factors[j] for j in job_ids], dtype=np.float64)
        self._isolated_policy._num_workers = self._num_workers
        iso = (throughputs * self._isolated_policy._alloc(throughputs, sf)).sum(axis=1)
        # stateful bookkeeping, finish_time_fairness.py:103-145
        for i, j in enumerate(job_ids):
            if j not in self._cumulative_isolated_time:
                self._cumulative_isolated_time[j] = 0
            if j in self._num_steps_remaining_prev_iteration:
                self._cumulative_isolated_time[j] += (
                    self._num_steps_remaining_prev_iteration[j] - num_steps_remaining[j]
                ) / self._isolated_throughputs_prev_iteration[j]
        n = np.array([num_steps_remaining[j] for j in job_ids], dtype=np.float64)
        t = np.array([times_since_start[j] for j in job_ids], dtype=np.float64)
        den = np.array([self._cumulative_isolated_time[j] for j in job_ids], dtype=np.float64) + n / iso
        if thr is None:
            x2, self.last_objective, rc = self._solve_hetero(POL_FTF, throughputs, sf, t=t, n=n, den=den)
        else:
            x, self.last_objective, rc = _pooled(POL_FTF, N, thr, sf, t=t, n=n, den=den)
            x2 = self._split(x, share)
        self._num_steps_remaining_prev_iteration = copy.copy(num_steps_remaining)
        self._isolated_throughputs_prev_iteration = {j: iso[i] for i, j in enumerate(job_ids)}
        if rc != 0:     # "x.value is None" -> isolated allocation (finish_time_fairness.py:147-151)
            return self._isolated_policy.get_allocation(unflattened_throughputs, scale_factors, cluster_spec)
        return super().unflatten(x2, index)


class FinishTimeFairnessPolicy(Policy):
    def __init__(self, solver):
        self._name = "FinishTimeFairness"
        self._finish_time_fairness_perf_policy = FinishTimeFairnessPolicyWithPerf(solver)

    def get_allocation(self, unflattened_throughputs, scale_factors, unflattened_priority_weights,
                       times_since_start, num_steps_remaining, cluster_spec):
        throughputs, index = super().flatten(unflattened_throughputs, cluster_spec)
        if throughputs is None:
            return None
        v100 = {j: {w: unflattened_throughputs[j]["v100"] for w in unflattened_throughputs[j]}
                for j in unflattened_throughputs}       # finish_time_fairness.py:38-46
        return self._finish_time_fairness_perf_policy.get_allocation(
            v100, scale_factors, unflattened_priority_weights, times_since_start, num_steps_remaining, cluster_spec)


class MinTotalDurationPolicyWithPerf(Policy):
    def __init__(self, solver):
        Policy.__init__(self, solver)
        self._name = "MinTotalDuration_Perf"

    def get_allocation(self, unflattened_throughputs, scale_factors, num_steps_remaining, cluster_spec):
        throughputs, index = super().flatten(unflattened_throughputs, cluster_spec)
        if index is None:
            return None
        job_ids, _ = index
        thr, N, share = self._pool(throughputs)
        sf = np.array([scale_factors[j] for j in job_ids], dtype=np.float64)
        n = np.array([num_steps_remaining[j] for j in job_ids], dtype=np.float64)
        if thr is None:
            x2, self.last_objective, rc = self._solve_hetero(POL_MTD, throughputs, sf, n=n)
        else:
            x, self.last_objective, rc = _pooled(POL_MTD, N, thr, sf, n=n)
            x2 = self._split(x, share)
        assert rc == 0          # min_total_duration.py:132 `assert last_feasible_x is not None`
        return super().unflatten(x2, index)


class MinTotalDurationPolicy(Policy):
    def __init__(self, solver):
        self._name = "MinTotalDuration"
        self._min_total_duration_perf_policy = MinTotalDurationPolicyWithPerf(solver)

    def get_allocation(self, unflattened_throughputs, scale_factors, num_steps_remaining, cluster_spec):
        throughputs, index = super().flatten(unflattened_throughputs, cluster_spec)
        if throughputs is None:
            return None
        v100 = {j: {w: unflattened_throughputs[j]["v100"] for w in unflattened_throughputs[j]}
                for j in unflattened_throughputs}
        return self._min_total_duration_perf_policy.get_allocation(v100, scale_factors, num_steps_remaining,
                                                                   cluster_spec)


class ThroughputNormalizedByCostSumWithPerfSLOs(Policy):
    def __init__(self, solver):
        Policy.__init__(self, solver)
        self._name = "ThroughputNormalizedByCostSum_PerfSLOs"

    def get_allocation(self, unflattened_throughputs, scale_factors, cluster_spec, instance_costs=None, SLOs={},
                       num_steps_remaining={}):
        throughputs, index = super().flatten(unflattened_throughputs, cluster_spec)
        if throughputs is None:
            return None
        job_ids, worker_types = index
        thr, N, share = self._pool(throughputs)
        sf = np.array([scale_factors[j] for j in job_ids], dtype=np.float64)
        cost = np.ones(len(worker_types))
        if instance_costs is not None:
            cost = np.array([instance_costs[w] for w in worker_types], dtype=np.float64)
        live_cost = cost[np.asarray(self._num_workers) > 0]
        if thr is None or not np.allclose(live_cost, live_cost[0]):
            need = None
            if SLOs:    # max_sum_throughput.py:87-93: sum_w thr_jw x_jw >= num_steps_remaining_j / SLO_j
                need = np.zeros(len(job_ids))
                for job_id in SLOs:
                    assert job_id in num_steps_remaining
                    need[job_ids.index(job_id)] = num_steps_remaining[job_id] / SLOs[job_id]
            x, self.last_objective, rc = self._solve_hetero(POL_MAXSUM, throughputs / cost[None, :], sf, t=need,
                                                            den=None if need is None else live_cost)
            if rc != 0:     # the reference warns and solves again without the SLO rows (:100-104)
                print("WARNING: No allocation possible with provided SLOs!")
                x, self.last_objective, rc = self._solve_hetero(POL_MAXSUM, throughputs / cost[None, :], sf)
            return super().unflatten(x, index)
        lo = None
        if SLOs:        # max_sum_throughput.py:87-93: sum_w thr_jw x_jw >= num_steps_remaining_j / SLO_j
            lo = np.zeros(len(job_ids))
            for job_id in SLOs:
                i = job_ids.index(job_id)
                assert job_id in num_steps_remaining
                lo[i] = (num_steps_remaining[job_id] / SLOs[job_id]) / thr[i]
        x, self.last_objective, rc = _pooled(POL_MAXSUM, N, thr / live_cost[0], sf, t=lo)
        if rc != 0:     # "x.value is None": the reference warns and solves again without the SLO rows (:100-104)
            print("WARNING: No allocation possible with provided SLOs!")
            x, self.last_objective, rc = _pooled(POL_MAXSUM, N, thr / live_cost[0], sf)
        return super().unflatten(self._split(x, share), index)


class ThroughputSumWithPerf(Policy):
    def __init__(self, solver):
        self._name = "ThroughputSumWithPerf"
        self._policy = ThroughputNormalizedByCostSumWithPerfSLOs(solver)

    def get_allocation(self, unflattened_throughputs, scale_factors, cluster_spec):
        return self._policy.get_allocation(unflattened_throughputs, scale_factors, cluster_spec)


class ThroughputNormalizedByCostSumWithPerf(Policy):
    def __init__(self, solver):
        self._name = "ThroughputNormalizedByCostSum_Perf"
        self._policy = ThroughputNormalizedByCostSumWithPerfSLOs(solver)

    def get_allocation(self, unflattened_throughputs, scale_factors, cluster_spec, instance_costs):
        return self._policy.get_allocation(unflattened_throughputs, scale_factors, cluster_spec,
                                           instance_costs=instance_costs)


class AlloXPolicy(Policy):
    """allox.py:12-188: Hungarian-style min-cost assignment of the oldest unallocated jobs to (worker, queue
    position) slots; the assignment itself runs on the GPU (swb_allox_assign)."""

    def __init__(self, alpha=1.0):
        self._name = "AlloX_Perf"
        self._alpha = alpha
        self._prev_allocation = {}

    def get_allocation(self, unflattened_throughputs, scale_factors, times_since_start, num_steps_remaining,
                       per_round_schedule, cluster_spec):
        throughputs, index = super().flatten(unflattened_throughputs, cluster_spec)
        if throughputs is None:
            return None
        job_ids, worker_types = index
        prev = self._prev_allocation
        unalloc, already = [], []
        for job_id in unflattened_throughputs:                      # allox.py:46-60
            if job_id not in prev:
                unalloc.append(job_id)
            else:
                total = 0.0
                for w in worker_types:
                    total += prev[job_id][w]
                (already if total == 1.0 else unalloc).append(job_id)
        m = len(unalloc)
        n = 0
        w_of = {}
        for w in worker_types:                                      # allox.py:65-80
            num = cluster_spec[w]
            for j in already:
                if prev[j][w] == 1.0:
                    num -= 1
            for wid in range(n, n + num):
                w_of[wid] = w
                n += 1
        unalloc.sort(key=lambda x: -times_since_start[x])           # allox.py:101-104
        unalloc = unalloc[: max(int(self._alpha * m), n)]
        m = len(unalloc)
        allocation = {j: {w: 0.0 for w in cluster_spec} for j in job_ids}
        for j in job_ids:
            if j in prev:
                allocation[j] = copy.copy(prev[j])
        if m > 0 and n > 0:
            wt_index = {w: i for i, w in enumerate(worker_types)}
            p = np.zeros((m, len(worker_types)))
            for i, j in enumerate(unalloc):                          # allox.py:111-124
                for w in worker_types:
                    thr = unflattened_throughputs[j][w]
                    p[i, wt_index[w]] = num_steps_remaining[j] / (thr if thr != 0.0 else 1e-10)
            t = np.array([times_since_start[j] for j in unalloc], dtype=np.float64)
            wtype = np.array([wt_index[w_of[wid]] for wid in range(n)], dtype=np.int32)
            cols, self.last_objective = _engine().allox_assign(p, t, wtype)
            per_worker = {i: [] for i in range(n)}                   # allox.py:147-163
            for row, col in enumerate(cols):
                per_worker[int(col) % n].append((unalloc[row], int(col) // n))
            for wid in range(n):
                lst = [(x[0], len(per_worker[wid]) - 1 - x[1]) for x in per_worker[wid]]
                lst.sort(key=lambda x: x[1])
                if lst:
                    allocation[lst[0][0]][w_of[wid]] = 1.0 / scale_factors[lst[0][0]]
        self._prev_allocation = copy.copy(allocation)
        return allocation


class ShockwavePolicy(Policy):
    """Name holder, like scheduler/policies/shockwave.py:8-10."""
    def __init__(self):
        self._name = "shockwave"


def get_policy(policy_name, solver=None, seed=None, priority_reweighting_policies=None):
    """The GPU-backed subset of utils.get_policy (scheduler/utils.py:603-685)."""
    table = {
        "finish_time_fairness": lambda: FinishTimeFairnessPolicy(solver="GUROBI"),
        "finish_time_fairness_perf": lambda: FinishTimeFairnessPolicyWithPerf(solver=solver),
        "gandiva_fair": GandivProportionalPolicy, "isolated": IsolatedPolicy, "isolated_plus": IsolatedPlusPolicy,
        "max_min_fairness": lambda: MaxMinFairnessPolicy(solver=solver),
        "max_min_fairness_perf": lambda: MaxMinFairnessPolicyWithPerf(solver=solver),
        "max_min_fairness_water_filling": lambda: MaxMinFairnessWaterFillingPolicy(
            priority_reweighting_policies=priority_reweighting_policies),
        "max_min_fairness_water_filling_perf": lambda: MaxMinFairnessWaterFillingPolicyWithPerf(
            priority_reweighting_policies=priority_reweighting_policies),
        "max_sum_throughput_perf": lambda: ThroughputSumWithPerf(solver=solver),
        "max_sum_throughput_normalized_by_cost_perf": lambda: ThroughputNormalizedByCostSumWithPerf(solver=solver),
        "max_sum_throughput_normalized_by_cost_perf_SLOs": lambda: ThroughputNormalizedByCostSumWithPerfSLOs(solver=solver),
        "min_total_duration": lambda: MinTotalDurationPolicy(solver=solver),
        "min_total_duration_perf": lambda: MinTotalDurationPolicyWithPerf(solver=solver),
        "shockwave": ShockwavePolicy,
        # not in the reference's table (its strategy-proof classes are reachable by import only): names added here
        "max_min_fairness_strategy_proof": lambda: MaxMinFairnessStrategyProofPolicy(solver=solver),
        "max_min_fairness_strategy_proof_perf": lambda: MaxMinFairnessStrategyProofPolicyWithPerf(solver=solver),
    }
    packed = {"max_min_fairness_packed": "MaxMinFairnessPolicyWithPacking",
              "finish_time_fairness_packed": "FinishTimeFairnessPolicyWithPacking",
              "min_total_duration_packed": "MinTotalDurationPolicyWithPacking",
              "max_sum_throughput_normalized_by_cost_packed_SLOs": "ThroughputNormalizedByCostSumWithPackingSLOs"}
    if policy_name == "max_min_fairness_water_filling_packed":
        from . import packing
        return packing.MaxMinFairnessWaterFillingPolicyWithPacking(
            priority_reweighting_policies=priority_reweighting_policies)
    if policy_name in packed:       # the *_packed names of utils.py:626-672 (packing.py: LPs on swb_lp_solve)
        from . import packing
        return getattr(packing, packed[policy_name])(solver=solver)
    if policy_name.startswith("allox"):
        return AlloXPolicy(alpha=0.2 if policy_name == "allox" else float(policy_name.split("allox_alpha=")[1]))
    if policy_name not in table:
        raise ValueError("Unknown policy!")
    return table[policy_name]()
