"""P5 — closed loop: the UNMODIFIED reference simulator (scheduler/scheduler.py:1728-2268) driving the product's
ShockwaveScheduler / Gavel policies — libswb200.so in the loop — on the canonical 120-job trace
(reproduce/tacc_32gpus.sh), end-to-end metrics against the golden pickles the reference ships (within the 3 % spread of
its own three Shockwave pickles, BASELINE.md §2).

Needs a B200 AND the reference's simulator: the reference's scheduler/ directory, or the byte-compiled build of it that
build() makes under oracle/_ref/scheduler (git-ignored, `python -m oracle.stage_ref`).  Every run appends its metrics to
gpurun_out/closed_loop.json (copied to profiles/closed_loop_rNN.json for the record)."""
import glob
import json
import os
import pickle
import time

import numpy as np
import pytest

from oracle import ref_harness as rh

pytestmark = [pytest.mark.gpu, pytest.mark.reference]
GOLD = rh.GOLDEN_DIR
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _have_both():
    if not (os.path.isdir(rh.REF) and os.path.isdir(GOLD)):
        return False
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


def _record(name, out, gold, seconds, extra=None):
    ftf, gftf = np.array(out["finish_time_fairness_list"]), np.array(gold["finish_time_fairness_list"])
    row = dict(policy=name, seconds=round(seconds, 2),
               makespan=out["makespan"], golden_makespan=gold["makespan"],
               avg_jct=out["avg_jct"], golden_avg_jct=gold["avg_jct"],
               cluster_util=out["cluster_util"], golden_cluster_util=gold["cluster_util"],
               worst_ftf=float(ftf.max()), golden_worst_ftf=float(gftf.max()),
               unfair_fraction=float((ftf > 1.05).mean()), golden_unfair_fraction=float((gftf > 1.05).mean()),
               rounds=len(out["per_round_schedule"]), golden_rounds=len(gold["per_round_schedule"]))
    row.update(extra or {})
    d = os.path.join(ROOT, "gpurun_out")
    os.makedirs(d, exist_ok=True)
    path = os.path.join(d, "closed_loop.json")
    rows = json.load(open(path)) if os.path.exists(path) else []
    rows = [r for r in rows if r["policy"] != name] + [row]
    json.dump(rows, open(path, "w"), indent=1)
    return row


def _native_loaded():
    return any("libswb200.so" in line for line in open("/proc/self/maps"))


@pytest.mark.skipif(not _have_both(), reason="needs a B200 and the (staged) reference simulator at the same time")
def test_shockwave_closed_loop_matches_golden_pickle():
    from shockwave_b200 import ShockwaveScheduler
    stats = dict(solves=0, fallback=0, ms=0.0)

    class Counting(ShockwaveScheduler):
        def _resolve(self, jobids, jobobjs):
            t0 = time.perf_counter()
            out = super()._resolve(jobids, jobobjs)
            stats["ms"] += (time.perf_counter() - t0) * 1e3
            stats["solves"] += 1
            stats["fallback"] += int(self.last_result["status"] != 0)
            return out

    t0 = time.perf_counter()
    out = rh.simulate("shockwave", shockwave_scheduler_cls=Counting)
    assert _native_loaded() and stats["solves"] > 50
    gold = pickle.load(open(glob.glob(os.path.join(GOLD, "shockwave_*"))[0], "rb"))
    row = _record("shockwave", out, gold, time.perf_counter() - t0,
                  dict(resolves=stats["solves"], fallback_resolves=stats["fallback"],
                       mean_resolve_ms=stats["ms"] / max(1, stats["solves"])))
    print(row)
    assert abs(out["makespan"] - gold["makespan"]) / gold["makespan"] < 0.03
    assert abs(out["avg_jct"] - gold["avg_jct"]) / gold["avg_jct"] < 0.03
    assert abs(out["cluster_util"] - gold["cluster_util"]) / gold["cluster_util"] < 0.03
    ftf, gftf = np.array(out["finish_time_fairness_list"]), np.array(gold["finish_time_fairness_list"])
    assert abs(ftf.max() - gftf.max()) / gftf.max() < 0.10
    assert abs((ftf > 1.05).mean() - (gftf > 1.05).mean()) < 0.03


def _pin(G):
    return os.path.join(ROOT, "tests", "golden", f"scale{G}_oracle_pin.json")


@pytest.mark.skipif(not _have_both(), reason="needs a B200 and the (staged) reference simulator at the same time")
@pytest.mark.parametrize("G", [64, 128, 256])
def test_shockwave_closed_loop_scale_runs_match_oracle_pins(G):
    """Closed-loop cases at the reference's scale-out sizes: the traces of reproduce/scale_{64,128,256}gpus.sh (220 / 460 /
    900 jobs; configurations/scale_*gpus.json: k = 10 / 1e-3 / 1e5, lambda = 5 / 15 / 5; wisr_throughputs.json).  The
    reference ships no golden pickles for them; the yardstick is the same unmodified simulator with the HiGHS oracle in
    place of Gurobi (tests/golden/make_scale_pins.py).  Same 3 % tolerance as the canonical case."""
    from shockwave_b200 import ShockwaveScheduler
    if not os.path.exists(_pin(G)):
        pytest.skip(f"no oracle pin recorded for the {G}-GPU run (tests/golden/make_scale_pins.py {G})")
    pin = json.load(open(_pin(G)))
    if not os.path.exists(os.path.join(rh.REF, pin["trace"])):
        pytest.skip("trace not staged")
    stats = dict(solves=0, fallback=0, ms=0.0, jmax=0)

    class Counting(ShockwaveScheduler):
        def _resolve(self, jobids, jobobjs):
            t0 = time.perf_counter()
            out = super()._resolve(jobids, jobobjs)
            stats["ms"] += (time.perf_counter() - t0) * 1e3
            stats["solves"] += 1
            stats["fallback"] += int(self.last_result["status"] != 0)
            stats["jmax"] = max(stats["jmax"], len(jobids))
            return out

    t0 = time.perf_counter()
    out = rh.simulate("shockwave", shockwave_scheduler_cls=Counting, config=pin["config"], cluster=pin["cluster"],
                      trace=pin["trace"], throughputs=pin["throughputs"])
    assert _native_loaded() and stats["solves"] > 50
    ftf = np.array(out["finish_time_fairness_list"])
    gold = dict(makespan=pin["makespan"], avg_jct=pin["avg_jct"], cluster_util=pin["cluster_util"],
                finish_time_fairness_list=[pin["worst_ftf"]] + [0.0] * (len(ftf) - 1),
                per_round_schedule=[None] * pin["rounds"])
    row = _record(f"shockwave@{G}gpus(vs oracle pin)", out, gold, time.perf_counter() - t0,
                  dict(resolves=stats["solves"], fallback_resolves=stats["fallback"], max_live_jobs=stats["jmax"],
                       mean_resolve_ms=stats["ms"] / max(1, stats["solves"]),
                       golden_unfair_fraction=pin["unfair_fraction"]))
    print(row)
    assert abs(out["makespan"] - pin["makespan"]) / pin["makespan"] < 0.03
    assert abs(out["avg_jct"] - pin["avg_jct"]) / pin["avg_jct"] < 0.03
    assert abs(out["cluster_util"] - pin["cluster_util"]) / pin["cluster_util"] < 0.03
    assert ftf.max() <= pin["worst_ftf"] * 1.10
    assert (ftf > 1.05).mean() <= pin["unfair_fraction"] + 0.03


@pytest.mark.skipif(not _have_both(), reason="needs a B200 and the (staged) reference simulator at the same time")
@pytest.mark.parametrize("policy", ["max_min_fairness", "finish_time_fairness", "min_total_duration",
                                    "max_sum_throughput_perf", "allox", "gandiva_fair"])
def test_gavel_policy_closed_loop_matches_golden_pickle(policy):
    from shockwave_b200 import policies
    t0 = time.perf_counter()
    out = rh.simulate(policy, policy_obj=policies.get_policy(policy, solver="ECOS", seed=0))
    assert _native_loaded()
    gold = pickle.load(open(glob.glob(os.path.join(GOLD, policy + "_120_*"))[0], "rb"))
    print(_record(policy, out, gold, time.perf_counter() - t0))
    # LP optima are degenerate in x; with the interior-point selection the HiGHS-backed run of the same host code
    # is within 0.8 % (tests/golden/tacc32_policy_pins.json), the GPU-backed one must be too
    assert abs(out["makespan"] - gold["makespan"]) / gold["makespan"] < 0.015
    assert abs(out["avg_jct"] - gold["avg_jct"]) / gold["avg_jct"] < 0.015


@pytest.mark.skipif(not _have_both(), reason="needs a B200 and the (staged) reference simulator at the same time")
@pytest.mark.parametrize("G", [64, 128, 256])
@pytest.mark.parametrize("policy", ["max_min_fairness", "finish_time_fairness", "min_total_duration"])
def test_gavel_policy_closed_loop_scale_runs_match_oracle_pins(policy, G):
    """The Gavel policies of BASELINE config E closed loop at the reference's scale-out sizes (220 / 460 / 900 jobs on
    64 / 128 / 256 GPUs, up to ~840 live jobs per get_allocation()): same host code, device kernels vs the HiGHS backend
    (tests/golden/make_scale_policy_pins.py), same tolerance as the canonical case."""
    from shockwave_b200 import policies
    pins = json.load(open(os.path.join(ROOT, "tests", "golden", "scale_policy_pins.json")))
    pin = pins.get(f"{policy}@{G}")
    if pin is None or not os.path.exists(os.path.join(rh.REF, pin["trace"])):
        pytest.skip("no pin / trace not staged")
    t0 = time.perf_counter()
    out = rh.simulate(policy, policy_obj=policies.get_policy(policy, solver="ECOS", seed=0), cluster=pin["cluster"],
                      trace=pin["trace"], throughputs=pin["throughputs"])
    assert _native_loaded()
    ftf = np.array(out["finish_time_fairness_list"])
    gold = dict(makespan=pin["makespan"], avg_jct=pin["avg_jct"], cluster_util=pin["cluster_util"],
                finish_time_fairness_list=[pin["worst_ftf"]] + [0.0] * (len(ftf) - 1),
                per_round_schedule=[None] * pin["rounds"])
    print(_record(f"{policy}@{G}gpus(vs oracle pin)", out, gold, time.perf_counter() - t0,
                  dict(golden_unfair_fraction=pin["unfair_frac"])))
    assert abs(out["makespan"] - pin["makespan"]) / pin["makespan"] < 0.015
    assert abs(out["avg_jct"] - pin["avg_jct"]) / pin["avg_jct"] < 0.015


@pytest.mark.skipif(not _have_both(), reason="needs a B200 and the (staged) reference simulator at the same time")
@pytest.mark.parametrize("policy", ["max_min_fairness", "finish_time_fairness", "max_sum_throughput_perf"])
def test_gavel_round_step_on_the_device_reproduces_the_reference_loop(policy):
    """§8(f)-2: priorities -> selection -> worker assignment of every round computed by gavel.cu (GavelRoundMixin in
    front of the reference's Scheduler class) — per_round_schedule must be identical, worker id by worker id, to the
    same run with the reference's own dict code."""
    from shockwave_b200 import policies
    from shockwave_b200.placement import GavelRoundMixin
    before = GavelRoundMixin.swb_round_calls
    t0 = time.perf_counter()
    dev = rh.simulate(policy, policy_obj=policies.get_policy(policy, solver="ECOS", seed=0),
                      scheduler_mixin=GavelRoundMixin)
    t_dev = time.perf_counter() - t0
    ncalls = GavelRoundMixin.swb_round_calls - before
    ref = rh.simulate(policy, policy_obj=policies.get_policy(policy, solver="ECOS", seed=0))
    assert ncalls == len(dev["per_round_schedule"]) > 100 and _native_loaded()
    assert len(dev["per_round_schedule"]) == len(ref["per_round_schedule"])
    for r, (a, b) in enumerate(zip(dev["per_round_schedule"], ref["per_round_schedule"])):
        assert list(a.items()) == list(b.items()), r
    assert dev["makespan"] == ref["makespan"] and dev["jct_list"] == ref["jct_list"]
    gold = pickle.load(open(glob.glob(os.path.join(GOLD, policy + "_120_*"))[0], "rb"))
    print(_record(policy + "+round_step_on_device", dev, gold, t_dev, dict(device_round_calls=ncalls)))
