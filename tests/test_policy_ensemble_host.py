"""Host logic of shockwave_b200.simulate.PolicyEnsemble (Gavel policies on the device round loop) against the UNMODIFIED
reference loop (CPU): the same policy code with the HiGHS backend behind it ran (a) inside the reference's
Scheduler.simulate() (recorded by tests/golden/make_loop_records.py) and runs (b) inside the ensemble driver, on the host
build of the device loop with the oracle restatement of the round step.  Identical per-round schedules (jobs AND worker
ids), completion times and makespan mean the driver keeps the Gavel time accounting, deficits, allocation-update triggers
and policy arguments exactly as scheduler.py:3205-3355, :3498-3551, :3611-3724, :4660-4672 do."""
import numpy as np
import pytest

from oracle import gavel_backend as gb
from oracle.gavel_round_backend import OracleBackend
from tests import sim_fixtures as sf_
from tests.golden import make_loop_records as records


@pytest.mark.parametrize("policy,keep,ngpus,static", [("max_min_fairness", 40, 12, True), ("max_min_fairness", 60, 12, False),
                                                       ("finish_time_fairness", 40, 8, False), ("min_total_duration", 40, 8, False),
                                                       ("isolated", 30, 8, True), ("max_sum_throughput_perf", 40, 8, False)])
def test_policy_ensemble_equals_the_reference_loop(monkeypatch, policy, keep, ngpus, static):
    if sf_.host_sim_lib() is None:
        pytest.skip("g++ not available")
    from shockwave_b200 import simulate as sim
    rec = records.load("policy", policy, keep, ngpus, static)
    with gb.cpu_backend() as P:
        monkeypatch.setattr(sim, "DeviceSim", sf_.HostDeviceSim)
        tr = {k: np.asarray(rec[k]) for k in ("arrival", "total_steps", "scale_factor", "throughput", "duration", "batch_size",
                                              "dataset_len")}
        ens = sim.PolicyEnsemble(tr, [P.get_policy(policy, solver="ECOS", seed=0) for _ in range(2)], ngpus,
                                 dynamic=None if static else rec["dyn"], round_backend=OracleBackend())
        out = ens.run()
    d = ens.result_dicts(rec["isolated"])[0]
    assert d["finish_time_fairness_list"] == rec["finish_time_fairness_list"]
    assert d["utilization_list"] == rec["utilization_list"] and d["cluster_util"] == rec["cluster_util"]
    assert [d["extension_percentage"], d["num_lease_extensions"], d["num_lease_extension_opportunities"]] == rec["lease"]
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
