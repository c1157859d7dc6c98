"""Host logic of shockwave_b200.simulate.PolicyEnsemble on MIXED clusters (several worker types, static jobs) against the
UNMODIFIED reference loop (CPU): the same policy code with the HiGHS backend behind it ran (a) inside the reference's
Scheduler.simulate() on a v100 + p100 + k80 cluster (recorded by tests/golden/make_loop_records.py) and runs (b) inside
the ensemble driver, on the host build of the device loop with the oracle restatement of the round step.  Identical
per-round schedules (jobs AND worker ids, same insertion order), completion times and makespan mean the driver keeps the
per-worker-type time accounting, deficits, worker-id layout and the order the types are walked in (incl. the reference's
type shuffler for the policies without `Perf` in their name) exactly as scheduler.py:1290-1301, :1826-1832, :3498-3551,
:3611-3724, :4660-4672 do."""
import numpy as np
import pytest

from oracle import gavel_backend as gb
from oracle import sim_loop
from oracle.gavel_round_backend import OracleBackend
from tests import sim_fixtures as sf_
from tests.golden import make_loop_records as records


@pytest.mark.parametrize("policy,keep,cluster", [("max_min_fairness_perf", 40, "4:3:2"), ("finish_time_fairness_perf", 36, "2:4:4"),
                                                  ("max_min_fairness", 40, "4:3:2"), ("min_total_duration_perf", 30, "4:0:4"),
                                                  ("max_sum_throughput_perf", 30, "4:2:4")])
def test_policy_ensemble_on_a_mixed_cluster_equals_the_reference_loop(monkeypatch, policy, keep, cluster):
    if sf_.host_sim_lib() is None:
        pytest.skip("g++ not available")
    from shockwave_b200 import simulate as sim
    rec = records.load("hetero", policy, keep, cluster)
    tr = sim_loop.trace_arrays(rec)
    wt = dict(names=rec["worker_types"], throughput=np.asarray(rec["throughput_w"]), ngpus=rec["ngpus_w"])
    with gb.cpu_backend() as P:
        monkeypatch.setattr(sim, "DeviceSim", sf_.HostDeviceSim)
        ens = sim.PolicyEnsemble(tr, [P.get_policy(policy, solver="ECOS", seed=0) for _ in range(2)], None,
                                 worker_types=wt, round_backend=OracleBackend(), seed=0)
        out = ens.run()
    want = [{j: tuple(ws) for j, ws in rnd} for rnd in rec["per_round_workers"]]
    for s in (0, 1):
        got = out["per_round_schedule"][s]
        first = next((i for i in range(min(len(got), len(want))) if got[i] != want[i]), None)
        assert first is None and len(got) == len(want), (first, got[first] if first is not None else None,
                                                        want[first] if first is not None else None)
        assert [list(r) for r in got] == [list(r) for r in want]            # same insertion order too
        assert out["makespan"][s] == rec["makespan"] and out["rounds"][s] == rec["rounds"]
        for j in range(keep):
            assert out["jct"][s, j] == rec["jct"][str(j)]
    assert len({w for rnd in rec["per_round_schedule"] for _, w in rnd}) == len(rec["ngpus_w"])   # every type was used
