"""Host logic of shockwave_b200.simulate.ShockwaveEnsemble against the UNMODIFIED reference loop (CPU): the same
deterministic stand-in scheduler (a rule on the arrays a re-solve uploads: epoch progress, timeline summaries, submit
times, round pointer) ran (a) inside the reference's Scheduler.simulate() (recorded by tests/golden/make_loop_records.py)
and runs (b) inside the ensemble driver on the host build of the device round loop.  Identical per-round schedules,
completion times and makespan mean the driver maintains the scheduler state exactly as scheduler.py:1878-2375 does
(metadata add / remove order, resolve triggers, round pointer, REOPT_ROUNDS, progress and timeline updates)."""
import os
import tempfile

import numpy as np
import pytest

from tests import sim_fixtures as sf_
from tests.golden import make_loop_records as records


@pytest.mark.parametrize("keep,ngpus,static", [(24, 8, True), (60, 16, True), (60, 16, False), (120, 32, False)])
def test_ensemble_driver_equals_the_reference_loop(monkeypatch, keep, ngpus, static):
    if sf_.host_sim_lib() is None:
        pytest.skip("g++ not available")
    from shockwave_b200 import simulate as sim
    scratch = tempfile.mkdtemp(prefix="swens_")
    rec = records.load("shockwave", keep, ngpus, static)
    cfg = rec["config"]
    Rule = sf_.make_rule_scheduler_cls()
    # ---- the ensemble on the host build, two identical scenarios + one with another window length
    ens_log = []
    Rule.log = ens_log
    monkeypatch.setattr(sim, "DeviceSim", sf_.HostDeviceSim)
    monkeypatch.setattr(sim, "ShockwaveScheduler", Rule)
    tr = {k: np.asarray(rec[k]) for k in ("arrival", "total_steps", "scale_factor", "throughput", "duration", "batch_size",
                                          "dataset_len")}
    ens = sim.ShockwaveEnsemble(tr, rec["profiles"], cfg, [{}, {}, {"future_rounds": cfg["future_rounds"] + 3}],
                                ngpus=ngpus, time_per_iteration=120, dynamic=None if static else rec["dyn"])
    Rule.log = None
    out = ens.run()
    want = rec["per_round_jobs"]
    for s in (0, 1):
        assert out["per_round_schedule"][s] == want
        assert out["makespan"][s] == rec["makespan"] and out["rounds"][s] == rec["rounds"]
        for j in range(keep):
            assert out["jct"][s, j] == rec["jct"][str(j)]
    assert np.isfinite(out["jct"][2]).all()
    # the result dict of a scenario against what the reference computes from its own run (scheduler.py:2779-2925, :3037-3058)
    d = ens.result_dicts()[0]
    assert d["finish_time_fairness_list"] == rec["finish_time_fairness_list"]
    assert d["jct_list"] == [rec["jct"][str(j)] for j in range(keep)]
    assert d["avg_jct"] == pytest.approx(rec["avg_jct"], rel=1e-12) and d["makespan"] == rec["makespan"]
    assert d["cluster_util"] == pytest.approx(rec["cluster_util"], abs=2e-5)
    paths = ens.write_result_pickles(os.path.join(scratch, "results"))
    import pickle
    assert pickle.load(open(paths[1], "rb"))["makespan"] == rec["makespan"]
