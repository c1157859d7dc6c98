"""Scenario sharding of the what-if ensemble over ranks (CPU, gloo, world size 2): every rank runs its slice on the
host build of the device loop with the rule scheduler, results are exchanged with all_gather_object; the merged result
equals the single-process run scenario by scenario."""
import os

import numpy as np
import pytest

from tests import sim_fixtures as sf_

CFG = {"future_rounds": 12, "k": 1e-3, "lambda": 12.0, "rhomax": 1.0, "log_approximation_bases": [0.0, 0.2, 0.4, 0.6, 0.8, 1.0]}
SCEN = [{}, {"future_rounds": 5}, {"future_rounds": 3}, {"future_rounds": 7}, {"future_rounds": 2}]


def _inputs():
    tr = sf_.random_trace(40, 11)
    tr["arrival"][0] = 0.0
    profiles = []
    for j in range(40):
        spe = int(np.ceil(tr["dataset_len"][j] / tr["batch_size"][j]))
        ep = int(np.ceil(tr["total_steps"][j] / spe))
        profiles.append(dict(scale_factor=int(tr["scale_factor"][j]), num_epochs=ep, num_samples_per_epoch=int(tr["dataset_len"][j]),
                             duration_every_epoch=[spe / tr["throughput"][j]] * ep, bs_every_epoch=[int(tr["batch_size"][j])] * ep))
    return tr, profiles


def _patch(set_=setattr):
    """CPU stand-ins for the device loop and the solver: `set_` is monkeypatch.setattr in the pytest process (undone
    after the test, so later GPU tests get the device classes back), plain setattr in a spawned rank."""
    from shockwave_b200 import simulate as sim
    set_(sim, "DeviceSim", sf_.HostDeviceSim)
    set_(sim, "ShockwaveScheduler", sf_.make_rule_scheduler_cls())
    return sim


def _worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    sim = _patch()
    tr, profiles = _inputs()

    def gather(obj):
        out = [None] * world
        dist.all_gather_object(out, obj)
        return out
    res = sim.run_sharded(tr, profiles, CFG, SCEN, 8, rank=rank, world=world, gather=gather, device=0)
    q.put((rank, res["makespan"], res["jct"], res["rounds"], res["per_round_schedule"]))
    dist.destroy_process_group()


def test_two_rank_sharded_sweep_equals_the_single_process_run(monkeypatch):
    if sf_.host_sim_lib() is None:
        pytest.skip("g++ not available")
    import torch.multiprocessing as tmp
    ctx = tmp.get_context("spawn")
    q = ctx.Queue()
    port = 31000 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted([q.get(timeout=300) for _ in range(2)], key=lambda t: t[0])
    for p in procs:
        p.join(timeout=60)
    sim = _patch(monkeypatch.setattr)
    tr, profiles = _inputs()
    one = sim.run_sharded(tr, profiles, CFG, SCEN, 8, device=0)
    assert sim.shard_scenarios(5, 0, 2) == [0, 2, 4] and sim.shard_scenarios(5, 1, 2) == [1, 3]
    for _, makespan, jct, rounds, sched in res:
        assert np.array_equal(makespan, one["makespan"]) and np.array_equal(rounds, one["rounds"])
        assert np.array_equal(jct, one["jct"], equal_nan=True)
        assert sched == one["per_round_schedule"]
    assert len({tuple(map(tuple, s)) for s in one["per_round_schedule"]}) > 1          # the what-ifs do differ


# ---- the same for the Gavel-policy ensembles (what-ifs = policies), on a mixed cluster ----
POLICIES = ["max_min_fairness_perf", "finish_time_fairness_perf", "max_min_fairness", "min_total_duration_perf",
            "max_sum_throughput_perf"]


def _policy_inputs():
    tr = sf_.random_trace(30, 5)
    tr["arrival"][0] = 0.0
    rng = np.random.default_rng(2)
    wt = dict(names=["k80", "p100", "v100"], ngpus=[4, 4, 5],
              throughput=tr["throughput"][:, None] * np.sort(rng.uniform(0.2, 1.0, (30, 3)), axis=1))
    return tr, wt


def _run_policies(rank, world, gather, set_=setattr):
    from oracle import gavel_backend as gb
    from oracle.gavel_round_backend import OracleBackend
    sim = _patch(set_)
    tr, wt = _policy_inputs()
    with gb.cpu_backend() as P:
        P.set_device = lambda d: None                      # no engine on the CPU stand-ins
        try:
            return sim.run_policies_sharded(tr, POLICIES, None, rank=rank, world=world, gather=gather, device=0,
                                            make_policy=lambda n: P.get_policy(n, solver="ECOS", seed=0),
                                            worker_types=wt, round_backend=OracleBackend())
        finally:
            del P.set_device


def _policy_worker(rank, world, port, q):
    import importlib

    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)

    def gather(obj):
        out = [None] * world
        dist.all_gather_object(out, obj)
        return out
    res = _run_policies(rank, world, gather)
    q.put((rank, res["makespan"], res["jct"], res["rounds"], res["per_round_schedule"]))
    dist.destroy_process_group()


def test_two_rank_sharded_policy_sweep_equals_the_single_process_run(monkeypatch):
    if sf_.host_sim_lib() is None:
        pytest.skip("g++ not available")
    import torch.multiprocessing as tmp
    ctx = tmp.get_context("spawn")
    q = ctx.Queue()
    port = 33000 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_policy_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted([q.get(timeout=300) for _ in range(2)], key=lambda t: t[0])
    for p in procs:
        p.join(timeout=60)
    one = _run_policies(0, 1, None, monkeypatch.setattr)
    assert np.isfinite(one["makespan"]).all()
    for _, makespan, jct, rounds, sched in res:
        assert np.array_equal(makespan, one["makespan"]) and np.array_equal(rounds, one["rounds"])
        assert np.array_equal(jct, one["jct"], equal_nan=True)
        assert sched == one["per_round_schedule"]
    assert len(set(one["makespan"].tolist())) > 1                                       # the policies do differ
