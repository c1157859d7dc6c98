"""Generator of tests/golden/loop_records.json.gz: the runs of the UNMODIFIED reference simulator (scheduler.py:1728-2268)
that the host tests of the ensemble drivers compare against, stored so that those tests need no copy of the reference.
One record per test case, holding what the test reads from the reference's run: the trace as plain arrays (+ the dynamic
tables, the job profiles), the per-round schedule with worker ids in the reference's insertion order, completion times,
makespan, rounds and the reference's result-pickle figures.

  policy     tests/test_policy_ensemble_host.py            Gavel policies, HiGHS backend, one worker type
  shockwave  tests/test_sim_ensemble_host.py               the rule scheduler of tests/sim_fixtures.py as the solver
  hetero     tests/test_policy_ensemble_hetero_host.py     mixed v100 + p100 + k80 clusters (make_sim_hetero_pins.record)

    python -m tests.golden.make_loop_records         (needs the reference's scheduler/ directory, see oracle/ref_harness.py)
"""
import gzip
import json
import os
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
PATH = os.path.join(ROOT, "tests", "golden", "loop_records.json.gz")

# the parameter sets of the three tests
POLICY_CASES = [("max_min_fairness", 40, 12, True), ("max_min_fairness", 60, 12, False),
                ("finish_time_fairness", 40, 8, False), ("min_total_duration", 40, 8, False),
                ("isolated", 30, 8, True), ("max_sum_throughput_perf", 40, 8, False)]
SHOCKWAVE_CASES = [(24, 8, True), (60, 16, True), (60, 16, False), (120, 32, False)]
HETERO_CASES = [("max_min_fairness_perf", 40, "4:3:2"), ("finish_time_fairness_perf", 36, "2:4:4"),
                ("max_min_fairness", 40, "4:3:2"), ("min_total_duration_perf", 30, "4:0:4"),
                ("max_sum_throughput_perf", 30, "4:2:4")]

_cache = {}


def key(kind, *case):
    return "/".join([kind] + [str(v) for v in case])


def load(kind, *case):
    if "d" not in _cache:
        with gzip.open(PATH, "rt") as f:
            _cache["d"] = json.load(f)
    return _cache["d"][key(kind, *case)]


def _workers(per_round_schedule):
    """[{job id: worker ids}] -> [[[job, [worker ids]], ...]] in the reference's dict insertion order."""
    return [[[int(k), [int(w) for w in v]] for k, v in rnd.items()] for rnd in per_round_schedule]


def _result_fields(ref, rec):
    rec.pop("timeline", None)                  # not read by the tests
    rec.update(makespan=float(ref["makespan"]), avg_jct=float(ref["avg_jct"]), cluster_util=float(ref["cluster_util"]),
               finish_time_fairness_list=[float(v) for v in ref["finish_time_fairness_list"]])
    return rec


def policy_case(policy, keep, ngpus, static):
    from oracle import gavel_backend as gb
    from oracle import ref_harness as rh
    from tests.golden import make_sim_pins as pins
    scratch = tempfile.mkdtemp(prefix="swpol_")
    pins.stage_static_trace(scratch, keep=keep, static=static)

    def extract(sched, jobs, arrival_times):
        rec = (pins.extract if static else pins.extract_dynamic)(sched, jobs, arrival_times)
        rec["lease"] = list(sched.get_num_lease_extensions(verbose=False))
        rec["isolated"] = [sum(sched._profiles[j]["duration_every_epoch"]) for j in range(len(jobs))]
        rec["utilization_list"] = [float(u) for u in sched.get_cluster_utilization()[1]]
        return rec
    with gb.cpu_backend() as P:
        ref = rh.simulate(policy, policy_obj=P.get_policy(policy, solver="ECOS", seed=0), trace=pins.REL, scratch=scratch,
                          cluster=f"{ngpus}:0:0", extract=extract)
    rec = _result_fields(ref, ref["extra"])
    rec["per_round_workers"] = _workers(ref["per_round_schedule"])
    return rec


def shockwave_case(keep, ngpus, static):
    from oracle import ref_harness as rh
    from tests import sim_fixtures as sf_
    from tests.golden import make_sim_pins as pins
    scratch = tempfile.mkdtemp(prefix="swens_")
    dst = pins.stage_static_trace(scratch, keep=keep, static=static)
    Rule = sf_.make_rule_scheduler_cls()

    def extract(sched, jobs, arrival_times):
        rec = (pins.extract if static else pins.extract_dynamic)(sched, jobs, arrival_times)
        rec["profiles"] = [dict(p) for p in sched._profiles[:len(jobs)]]
        return rec
    ref = rh.simulate("shockwave", shockwave_scheduler_cls=Rule, trace=pins.REL, scratch=scratch,
                      cluster=f"{ngpus}:0:0", extract=extract)
    rec = _result_fields(ref, ref["extra"])
    rec["per_round_jobs"] = [sorted(int(k) for k in rnd.keys()) for rnd in ref["per_round_schedule"]]
    rec["config"] = json.load(open(os.path.join(dst, "configurations/tacc_32gpus.json")))
    return rec


def hetero_case(policy, keep, cluster):
    from tests.golden import make_sim_hetero_pins as gen
    return gen.record(policy, keep, cluster)


def _plain(o):
    return o.item() if hasattr(o, "item") else o.tolist()


def main():
    out = {}
    for kind, cases, fn in (("policy", POLICY_CASES, policy_case), ("shockwave", SHOCKWAVE_CASES, shockwave_case),
                            ("hetero", HETERO_CASES, hetero_case)):
        for case in cases:
            out[key(kind, *case)] = fn(*case)
            print(key(kind, *case), out[key(kind, *case)]["makespan"], flush=True)
    with gzip.GzipFile(PATH, "wb", mtime=0) as f:
        f.write(json.dumps(out, default=_plain, separators=(",", ":")).encode())


if __name__ == "__main__":
    main()
