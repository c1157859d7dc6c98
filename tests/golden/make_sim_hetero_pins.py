"""Generator of tests/golden/sim_hetero_pins.json: the UNMODIFIED reference simulator (scheduler.py:1728-2268) on the
first jobs of the canonical trace (every job `static`) on MIXED clusters (v100 + p100 + k80 workers, the Gavel use case)
under heterogeneity-aware policies backed by the HiGHS oracle.  Recorded per run: the trace as plain arrays with the
per-worker-type throughputs [J][W] (W in the reference's sorted worker-type order k80, p100, v100), the per-round
schedule WITH the worker type every job ran on, and what the reference's bookkeeping made of it — completion times,
makespan, rounds.  oracle/sim_loop.py and the host build of sim_core.cuh replay the recorded schedules and must
reproduce these numbers exactly (tests/test_oracle_sim_hetero.py); the device loop does the same on the B200
(tests/test_zz_gpu_sim_hetero.py).

    python -m tests.golden.make_sim_hetero_pins         (needs the reference's scheduler/ directory or its build under oracle/_ref)
"""
import json
import os
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import gavel_backend as gb          # noqa: E402
from oracle import ref_harness as rh            # noqa: E402
from tests.golden import make_sim_pins as pins  # noqa: E402

RUNS = (("max_min_fairness_perf", 40, "4:3:2"), ("finish_time_fairness_perf", 36, "2:4:4"),
        ("max_min_fairness_perf", 60, "8:0:6"))


def extract(sched, jobs, arrival_times):
    rec = pins.extract(sched, jobs, arrival_times)
    types = sorted(sched._cluster_spec) if hasattr(sched, "_cluster_spec") else ["k80", "p100", "v100"]
    rec["worker_types"] = types
    rec["throughput_w"] = [[float(sched._oracle_throughputs[w][(j.job_type, j.scale_factor)]["null"]) for w in types]
                           for j in jobs]
    rec["worker_type_of_id"] = {str(k): types.index(v) for k, v in sched._worker_id_to_worker_type_mapping.items()}
    rec["ngpus_w"] = [sum(1 for v in sched._worker_id_to_worker_type_mapping.values() if v == w) for w in types]
    rec.pop("timeline", None)
    return rec


def record(policy, keep, cluster, scratch=None, product=False):
    """product=False: the reference loop as shipped with the HiGHS-backed policies (CPU).  product=True: the reference
    loop driving the PRODUCT's policies and round step on the device (GavelRoundMixin; needs a B200)."""
    scratch = scratch or tempfile.mkdtemp(prefix="swsimh_")
    pins.stage_static_trace(scratch, keep=keep, static=True)
    if product:
        from shockwave_b200 import policies as P
        from shockwave_b200.placement import GavelRoundMixin
        r = rh.simulate(policy, policy_obj=P.get_policy(policy, solver="ECOS", seed=0), trace=pins.REL, scratch=scratch,
                        cluster=cluster, extract=extract, scheduler_mixin=GavelRoundMixin)
    else:
        with gb.cpu_backend() as P:
            r = rh.simulate(policy, policy_obj=P.get_policy(policy, solver="ECOS", seed=0), trace=pins.REL,
                            scratch=scratch, cluster=cluster, extract=extract)
    rec = r["extra"]
    wt = rec["worker_type_of_id"]
    # {job: worker type index} per round, in the reference's dict insertion order
    rec["per_round_schedule"] = [[[int(k), wt[str(v[0])]] for k, v in rnd.items()] for rnd in r["per_round_schedule"]]
    rec["per_round_workers"] = [[[int(k), [int(x) for x in v]] for k, v in rnd.items()] for rnd in r["per_round_schedule"]]
    rec.update(makespan=float(r["makespan"]), avg_jct=float(r["avg_jct"]), cluster=cluster, policy=policy,
               time_per_iteration=120)
    return rec


def main():
    out = {}
    for policy, keep, cluster in RUNS:
        rec = record(policy, keep, cluster)
        out[f"{policy}_{keep}_{cluster}"] = rec
        print(policy, keep, cluster, rec["makespan"], rec["rounds"], rec["ngpus_w"], flush=True)
    with open(os.path.join(ROOT, "tests", "golden", "sim_hetero_pins.json"), "w") as f:
        json.dump(out, f)


if __name__ == "__main__":
    main()
