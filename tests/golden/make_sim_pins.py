"""Generator of tests/golden/sim_static_pins.json: the UNMODIFIED reference simulator (scheduler.py:1728-2268) on the
canonical 120-job trace with every job's adaptation mode set to `static` (the device round loop of
shockwave_b200/csrc/sim.cu covers static jobs only), under two solver-free / CPU-backed policies.  Recorded per run: the
trace as plain arrays, the per-round schedule the reference chose, and what the reference's bookkeeping made of it —
completion times, makespan, the measured-throughput timeline of every job (`_throughput_timeline`, scheduler.py:549-571).
The restatement oracle/sim_loop.py replays the recorded schedules and must reproduce these numbers exactly.

    python -m tests.golden.make_sim_pins         (needs the reference's scheduler/ directory or its build under oracle/_ref)
"""
import json
import math
import os
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import gavel_backend as gb          # noqa: E402
from oracle import ref_harness as rh            # noqa: E402

REL = "traces/reproduce/static120.trace"


def stage_static_trace(scratch, keep=None, static=True):
    dst = rh.prepare_tree(scratch)
    with open(os.path.join(dst, rh.CANONICAL_TRACE)) as f, open(os.path.join(dst, REL), "w") as g:
        for i, line in enumerate(f):
            if keep is not None and i >= keep:
                break
            p = line.rstrip("\n").split("\t")
            if static:
                p[7] = "static"
            g.write("\t".join(p) + "\n")
    return dst


def extract(sched, jobs, arrival_times):
    import utils as ref_utils                    # the reference's (imported by the harness)
    J = len(jobs)
    thr = []
    for j in jobs:
        key = (j.job_type, j.scale_factor)
        thr.append(float(sched._oracle_throughputs["v100"][key]["null"]))
    ds = [int(ref_utils.dataset_len[ref_utils.model_dataset_mapping[j.model]]) if hasattr(ref_utils, "dataset_len")
          else None for j in jobs]
    tl = {}
    for jid, od in sched._throughput_timeline.items():
        k = jid if isinstance(jid, int) else jid.integer_job_id()
        tl[str(k)] = [[int(r), float(v[0]), int(v[1])] for r, v in od.items()]
    jct = {}
    for jid, d in sched._job_completion_times.items():
        jct[str(jid.integer_job_id())] = float(d)
    return dict(arrival=[float(a) for a in arrival_times], total_steps=[int(j.total_steps) for j in jobs],
                scale_factor=[int(j.scale_factor) for j in jobs], batch_size=[int(j.batch_size) for j in jobs],
                dataset_len=ds, duration=[float(j.duration) for j in jobs], throughput=thr,
                timeline=tl, jct=jct, rounds=int(sched._num_completed_rounds))


def dynamic_inputs(jobs, sched):
    """What shockwave_b200.simulate.build_dynamic_tables needs beside the static arrays, taken from the reference."""
    import utils as ref_utils
    models = [j.model for j in jobs]
    modes = [j.mode for j in jobs]
    table = sched._oracle_throughputs["v100"]

    def throughput_of(model, bs, sf):
        key = (f"{model} (batch size {bs})", sf)
        return float(table[key]["null"]) if key in table else None
    return models, modes, throughput_of, ref_utils.get_gns_bs_pattern


def extract_dynamic(sched, jobs, arrival_times):
    from shockwave_b200.simulate import build_dynamic_tables
    rec = extract(sched, jobs, arrival_times)
    models, modes, thr_of, gns = dynamic_inputs(jobs, sched)
    # the jobs have been rescaled by the time the run ends: the ORIGINAL batch sizes / step counts are the trace's
    rec["batch_size"] = [int(sched._original_bs[j._job_id]) for j in jobs]
    rec["total_steps"] = [int(sched._original_num_steps[j._job_id]) for j in jobs]
    rec["throughput"] = [thr_of(m, b, s) for m, b, s in zip(models, rec["batch_size"], rec["scale_factor"])]
    dyn = build_dynamic_tables(models, modes, rec, thr_of, gns)
    rec["models"], rec["modes"] = models, modes
    rec["dyn"] = {k: (v.tolist() if hasattr(v, "tolist") else v) for k, v in dyn.items()}
    return rec


def main_dynamic():
    """Same records on the canonical trace AS SHIPPED (59 accordion, 57 gns, 4 static jobs)."""
    scratch = tempfile.mkdtemp(prefix="swsimd_")
    rh.prepare_tree(scratch)
    out = {}
    for policy, ngpu in (("fifo", 32), ("max_min_fairness", 32), ("max_min_fairness", 12)):
        with gb.cpu_backend() as P:
            pol = P.get_policy(policy, solver="ECOS", seed=0) if policy != "fifo" else None
            r = rh.simulate(policy, policy_obj=pol, scratch=scratch, cluster=f"{ngpu}:0:0", extract=extract_dynamic)
        rec = r["extra"]
        rec.update(makespan=float(r["makespan"]), avg_jct=float(r["avg_jct"]), ngpus=ngpu, time_per_iteration=120,
                   per_round_schedule=[sorted(int(k) for k in rnd.keys()) for rnd in r["per_round_schedule"]])
        if out:                                   # the tables are the same for every run of the trace: keep them once
            rec.pop("dyn")
        out[f"{policy}_{ngpu}"] = rec
        print(policy, ngpu, rec["makespan"], rec["rounds"], len(rec["per_round_schedule"]))
    with open(os.path.join(ROOT, "tests", "golden", "sim_dynamic_pins.json"), "w") as f:
        json.dump(out, f)


def main():
    scratch = tempfile.mkdtemp(prefix="swsim_")
    stage_static_trace(scratch)
    out = {}
    for policy, ngpu in (("fifo", 32), ("max_min_fairness", 32), ("max_min_fairness", 12)):
        with gb.cpu_backend() as P:
            pol = P.get_policy(policy, solver="ECOS", seed=0) if policy != "fifo" else None
            r = rh.simulate(policy, policy_obj=pol, trace=REL, scratch=scratch, cluster=f"{ngpu}:0:0", extract=extract)
        rec = r["extra"]
        rec.update(makespan=float(r["makespan"]), avg_jct=float(r["avg_jct"]), ngpus=ngpu, time_per_iteration=120,
                   per_round_schedule=[sorted(int(k) for k in rnd.keys()) for rnd in r["per_round_schedule"]])
        out[f"{policy}_{ngpu}"] = rec
        print(policy, ngpu, rec["makespan"], rec["rounds"], len(rec["per_round_schedule"]))
    with open(os.path.join(ROOT, "tests", "golden", "sim_static_pins.json"), "w") as f:
        json.dump(out, f)


if __name__ == "__main__":
    if sys.argv[1:] == ["dynamic"]:
        main_dynamic()
    else:
        main()
