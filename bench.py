#!/usr/bin/env python
"""bench.py — schedule rounds/sec of the per-round market solve on B200 (BASELINE.json metric).

Workload (identical in both arms, `config`): BASELINE config D — ONE re-solve per step of a 4096-job x 512-GPU x
64-round planning window, scenario `i` = tests/synth.py seeded with 1000 + i (+ rank offset), k cycling through the
shipped configurations' values.  That is SURVEY.md §8(d)'s metric: 1 / time of one full round_schedule() re-solve.

--impl ours (default)
  value   one step = Monte-Carlo (GBM, 8192 paths/job) forecast of the step's job set -> its mean replaces the
          deterministic remaining runtime ON THE DEVICE (swb_gbm_ensemble, z = 0) -> market solve (8-CTA cluster) ->
          round placement + back-fill, everything resident in HBM, CUDA events on the launching stream.
  e2e     the drop-in class itself: ShockwaveScheduler(forecast="gbm").round_schedule() with a forced re-solve per step
          (host packing, host->device copies of the per-call inputs, forecast + GBM + solve + placement on the device,
          device->host copies of the round masks, list building) — the call scheduler/scheduler.py:1131 makes.
  batched a second, clearly separated figure: S = 296 what-if scenarios (k x rhomax x forecast quantile) of one job
          set per step, one CTA each — the GBM forecast is computed once, path-sharded over the ranks with ONE NCCL
          all-reduce, and every scenario plans against its own quantile of that forecast.
  N > 1   independent scenario streams per rank (a single solve does not shard: "replicas only"), no data-path
          collective in the headline step; the only collective of the timed region is the max over ranks.

--impl reference
  the reference's own CPU path for the same steps: the HiGHS restatement of its MILP (oracle/shockwave_milp.py; Gurobi
  and cvxpy cannot be installed here), same seeds, same step count.  The reference's 15 s TimeLimit does not yield an
  incumbent at this size (recorded in round 1), so the limit is lifted until HiGHS returns a schedule within the
  reference's MIPGap 1e-3 (~2-5 min per scenario on one core); the K timed steps run concurrently, one single-threaded
  HiGHS process per step on K host cores (HiGHS' branch and bound is single-threaded).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BASES = [0.0, 0.2, 0.4, 0.6, 0.8, 1.0]
ORIGIN = {0.0: 1e-6}
J, G, T, D = 4096, 512, 64, 120.0
K_SWEEP = [1e-3, 1e1, 1e5]          # the k values of the shipped configurations/*.json
METRIC = "schedule rounds/sec (4096 jobs x 512 GPUs x 64-round window)"
# identical in both arms (the driver compares it): what ONE step is
CONFIG = {"workload": "BASELINE config D: 4096 jobs x 512 GPUs x 64-round window, one full re-solve per step",
          "scenario_of_step_i": "tests/synth.py synth_problem(4096, 512, 64, seed=1000+i+1000003*rank, "
                                "tight=3.0 if i % 4 else 0.5), k = [1e-3, 1e1, 1e5][i % 3], lam=12, rhomax=1",
          "scenarios_per_step": 1, "parallelism": "one scenario stream per rank (replicas), no data-path collective"}


def scenario(i, rank=0):
    from tests.synth import synth_problem
    pb = synth_problem(J, G, T, D, seed=1000 + i + 1000003 * rank, tight=3.0 if i % 4 else 0.5)
    return pb, K_SWEEP[i % len(K_SWEEP)]


class ClockSampler(threading.Thread):
    """SM clock / throttle reasons DURING the timed region, through NVML every 2 ms (the recipe's nvidia-smi fields)."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.sm, self.mx, self.power = index, False, [], None, []
        self.t0, self.t1, self.ts, self.bits = None, None, [], []

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[self.index]) if vis and vis.split(",")[self.index].isdigit() else self.index
            h = nv.nvmlDeviceGetHandleByIndex(phys)
            self.mx = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            while not self.stop_flag:
                self.ts.append(time.perf_counter())
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                try:
                    self.power.append(nv.nvmlDeviceGetPowerUsage(h) / 1000.0)
                    self.bits.append(int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)))
                except Exception:
                    self.power.append(0.0); self.bits.append(0)
                time.sleep(0.002)
        except Exception:
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", "--query-gpu=clocks.sm,clocks.max.sm",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5)
                a, b = [float(v) for v in out.stdout.strip().split(",")]
                self.sm.append(a); self.mx = b
            except Exception:
                pass

    def summary(self):
        idx = [i for i, t in enumerate(self.ts) if self.t0 is not None and self.t0 <= t <= (self.t1 or 1e300)]
        if not idx:
            idx = list(range(len(self.sm)))
        sm = [self.sm[i] for i in idx]
        reasons = set()
        for i in idx:
            if i < len(self.bits):
                for b, name in self.REASONS.items():
                    if self.bits[i] & b:
                        reasons.add(name)
        pw = [self.power[i] for i in idx if i < len(self.power)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": self.mx,
                "reasons": sorted(reasons), "samples": len(sm), "power_w_max": max(pw) if pw else None}


# ------------------------------------------------------------------------------------------ reference arm
def _ref_step(args):
    """One step on one host core: the HiGHS restatement of dynamic_eisenberg_gale_scheduling (model build + MILP at
    the reference's MIPGap + fallback priorities / second solve when the FTF rows are infeasible) + construct_schedules.
    `limit`: HiGHS time limit per MILP (the reference's own is 15 s)."""
    i, limit, do_rank = args
    from oracle import shockwave_milp as om
    logv = om.pwl_log_values(BASES, ORIGIN)
    pb, k = scenario(i)
    t0 = time.perf_counter()
    try:
        out = om.dynamic_eisenberg_gale(pb["g"], pb["E"], pb["c"], pb["dbar"], pb["rem"], pb["ftobj"], G, T, D,
                                        pb["round_ptr"], k, 12.0, 1.0, BASES, logv, rel_gap=1e-3, time_limit=limit,
                                        do_rank=do_rank)
        om.construct_schedules(out["x"], list(range(J)), pb["g"], pb["rem"], pb["round_ptr"], G)
        ok, status = True, int(out["status"])
    except AssertionError:      # "relaxed problem must have a solution" = no incumbent inside the limit
        ok, status = False, -1
    return ok, status, time.perf_counter() - t0


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp
    K, W = args.steps, args.warmup
    ncpu = os.cpu_count() or 1
    procs = max(1, min(K, ncpu, args.ref_procs))
    limit = args.ref_time_limit
    ctx = mp.get_context("spawn")
    with ctx.Pool(procs) as pool:
        # warm-up: the same code path with the reference's own 15 s limit (imports, model build, HiGHS start-up)
        t0 = time.perf_counter()
        warm = pool.map(_ref_step, [(i, 15.0, False) for i in range(W)]) if W > 0 else []
        warm_s = time.perf_counter() - t0
        t0 = time.perf_counter()
        out = pool.map(_ref_step, [(W + i, limit, False) for i in range(K)], chunksize=1)
        total = time.perf_counter() - t0
    solved = sum(1 for o in out if o[0])
    val = K / total
    per = [round(o[2], 1) for o in out]
    sample = (f"{K} timed steps = {K} config-D scenarios (seeds {1000 + W}..{1000 + W + K - 1}), {procs} concurrent "
              f"single-threaded HiGHS processes (scipy.optimize.milp, mip_rel_gap=1e-3 as in the reference; time limit "
              f"lifted from the reference's 15 s to {limit:.0f} s per MILP because 15 s yields no incumbent at this size); "
              f"schedules produced: {solved}/{K}; fallback path taken: {sum(1 for o in out if o[1] == 1)}/{K}; "
              f"seconds per scenario (one core each, concurrent): min {min(per)} median {float(np.median(per))} max {max(per)}; "
              f"the re-rank MILP of the fallback path (shockwave.py:714-793) is NOT included; warm-up: {W} steps with "
              f"the 15 s limit, {sum(1 for o in warm if o[0])}/{W} produced a schedule, {warm_s:.0f} s")
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "rounds/s", "n_gpus": args.gpus,
            "steps": K, "warmup": W, "ms_per_step": 1e3 * total / K, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": CONFIG,
            "solver": "HiGHS via scipy.optimize.milp — stand-in for Gurobi (not installable here: no package, no licence, "
                      "no network)",
            "incumbents": solved,
            "cpu_baseline": {"value": val, "unit": "rounds/s", "cores": procs, "kind": "port", "sample": sample,
                             "host_cores": ncpu},
            "e2e": {"value": val, "unit": "rounds/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------ ours
class _Job:      # what scheduler.py hands over (scheduler/JobMetaData.py:41-98), duck-typed
    def __init__(self, pb, jid):
        from collections import OrderedDict
        E = int(pb["E"][jid])
        self.nworkers, self.epochs, self.epoch_nsamples = int(pb["g"][jid]), E, 50000
        dur = max(1.0, round(float(pb["dbar"][jid])))
        self.epoch_duration_preprofiled = [dur] * E
        self.bs_schedule = [32] * (E // 2) + [64] * (E - E // 2)
        self.timestamp_submit, self.gavel_round_duration = 0.0, D
        self.throughput_measurements = OrderedDict()
        self.epoch_progress, self.waiting_delay = int(pb["c"][jid]), 0

    def set_epoch_progress(self, c): self.epoch_progress = c
    def reset_waiting_delay(self): self.waiting_delay = 0
    def add_waiting_delay(self, d): self.waiting_delay += d


def _ncu_traffic(kernel_substr):
    """dram bytes per launch of a kernel from this round's committed ncu summary (profiles/ncu_kernels_r02.json,
    written by profiles/summarize.py from the .ncu-rep of the same command); None when there is no capture."""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "ncu_kernels_r02.json")))
        for name, row in d.items():
            if kernel_substr in name and row.get("dram_bytes") is not None:
                return float(row["dram_bytes"]), row
    except Exception:
        pass
    return None, None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--scenarios", type=int, default=296, help="batched block: scenarios per GPU per step (2 x 148 SMs)")
    ap.add_argument("--mc-paths", type=int, default=8192, help="GBM sample paths per job")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the batched / dense / policy legs")
    ap.add_argument("--ref-procs", type=int, default=32, help="reference arm: concurrent HiGHS processes")
    ap.add_argument("--ref-time-limit", type=float, default=450.0,
                    help="reference arm: HiGHS limit per MILP (s); measured on one core: 120-190 s per config-D scenario, 192 s for a "
                         "fallback scenario (two MILPs), so the whole arm ends within a few minutes")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed as DIR/<name>.npy (rank 0), to compare two builds")
    args = ap.parse_args()
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    from shockwave_b200 import Engine, ShockwaveScheduler, make_params
    from shockwave_b200.forecast_mc import path_range

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    # bind this rank's host threads to the CPUs of its GPU's NUMA node (pinned buffers are then allocated there)
    numa = None
    try:
        import pynvml as nv
        nv.nvmlInit()
        h = nv.nvmlDeviceGetHandleByIndex(local)
        words = (os.cpu_count() + 63) // 64
        mask = nv.nvmlDeviceGetCpuAffinity(h, words)
        cpus = [64 * wi + b for wi, wv in enumerate(mask) for b in range(64) if (int(wv) >> b) & 1]
        if cpus:
            os.sched_setaffinity(0, cpus)
            numa = f"{len(cpus)} cpus ({cpus[0]}..{cpus[-1]})"
    except Exception:
        pass
    eng = Engine(local)
    W = max(args.warmup, 3)
    K = args.steps
    P_MC = args.mc_paths
    est = torch.cuda.current_stream(dev)

    # ---- scenarios of all steps, resident in HBM (inputs of `value`) -----------------------------------------
    NS = W + K
    pbs = [scenario(i, rank) for i in range(NS)]
    st = lambda key, dt: torch.from_numpy(np.ascontiguousarray(np.stack([p[0][key] for p in pbs]).astype(dt))).to(dev)
    dten = dict(g=st("g", np.int32), E=st("E", np.int32), c=st("c", np.int32), dbar=st("dbar", np.float64),
                rem=st("rem", np.float64), ftobj=st("ftobj", np.float64))
    prms = [make_params(G, T, D, p[1], 12.0, 1.0, BASES, ORIGIN, round_ptr=p[0]["round_ptr"]) for p in pbs]
    rng = np.random.default_rng(12345 + rank)
    mc_mu = torch.from_numpy(rng.uniform(-1e-3, 1e-3, (NS, J))).to(dev)
    mc_sg = torch.from_numpy(rng.uniform(0.0, 0.05, (NS, J))).to(dev)
    mc_H = torch.minimum(dten["E"] - dten["c"], torch.tensor(256, dtype=torch.int32, device=dev)).contiguous()
    mc_out = torch.zeros((2, J), dtype=torch.float64, device=dev)
    rem_mc = torch.zeros((1, J), dtype=torch.float64, device=dev)
    xm = torch.zeros((1, J, 2), dtype=torch.int64, device=dev)
    bm = torch.zeros((1, J, 2), dtype=torch.int64, device=dev)
    nr = torch.zeros((1, J), dtype=torch.int32, device=dev)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)   # > 126 MB L2
    torch.cuda.synchronize()
    ptr = lambda t, i: t[i].data_ptr()
    launches = [0]

    def step_resident(i):
        """forecast (GBM) -> its mean becomes the remaining runtime -> solve -> place; all device-resident."""
        eng.gbm_forecast_device(J, ptr(dten["rem"], i), ptr(mc_H, i), ptr(mc_mu, i), ptr(mc_sg, i), P_MC, 0, 7 + i,
                                mc_out.data_ptr())
        eng.gbm_ensemble(1, J, P_MC, mc_out.data_ptr(), [0.0], rem_mc.data_ptr())
        res = eng.solve_device([prms[i]], J,
                               dict(g=ptr(dten["g"], i), E=ptr(dten["E"], i), c=ptr(dten["c"], i),
                                    dbar=ptr(dten["dbar"], i), rem=rem_mc.data_ptr(), ftobj=ptr(dten["ftobj"], i),
                                    bfkey=rem_mc.data_ptr()),
                               dict(xmask=xm.data_ptr(), bfmask=bm.data_ptr(), nrounds=nr.data_ptr()),
                               per_scenario_jobs=False)
        tm = eng.last_timings()
        launches[0] += 2 + 2 * tm["passes"]
        return res[0], tm

    sampler = ClockSampler(local)
    sampler.start()
    # forecast -> ensemble -> solve -> place queued back to back on the context's stream, ONE synchronisation at the end
    # of the solve call (SWB_OPT_ASYNC_AUX): no host round trip between the kernels of a step
    eng.set_option(8, 1)
    for i in range(W):
        step_resident(i)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    sampler.t0 = time.perf_counter()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    ksolve, kplace, nfb, shortf = [], [], 0, 0
    launches[0] = 0
    torch.cuda.synchronize()
    for i in range(K):
        flush.fill_(i)                          # L2 flush between timed iterations (not timed)
        torch.cuda.synchronize()
        ev[i][0].record(est)
        res, tm = step_resident(W + i)          # the solve call ends with a stream synchronize: the events bracket the step
        ev[i][1].record(est)
        ksolve.append(tm["ms_solve"]); kplace.append(tm["ms_place"])
        nfb += int(res["status"] == 1); shortf += int(res["shortfall"])
    torch.cuda.synchronize()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, res, rem_mc, xm, bm, nr)
    if world > 1:
        dist.barrier()
    eng.set_option(8, 0)
    total_ms = sum(a.elapsed_time(b) for a, b in ev)
    tt = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    total_ms = float(tt.item())
    value = world * K / (total_ms * 1e-3)
    gpu_launches = launches[0]
    # GBM kernel alone (device time of the library's own events)
    eng.gbm_forecast_device(J, ptr(dten["rem"], 0), ptr(mc_H, 0), ptr(mc_mu, 0), ptr(mc_sg, 0), P_MC, 0, 7,
                            mc_out.data_ptr())
    mc_ms = eng.last_timings()["ms_solve"]

    # ---- e2e: the drop-in class, forced re-solve per step, host buffers, copies inside -------------------------
    from collections import OrderedDict
    pb0 = pbs[0][0]
    sw = ShockwaveScheduler(ngpus=G, gram=16, init_metadata=OrderedDict(), future_nrounds=T, round_duration=int(D),
                            solver_preference=["GUROBI"], solver_rel_gap=1e-3, solver_num_threads=24, solver_timeout=15,
                            n_epoch_vars_max=64, logapx_bases=BASES, logapx_origin=ORIGIN, k=1e-3, lam=12.0, rhomax=1.0,
                            device=local, forecast="gbm", gbm_paths=P_MC, gbm_seed=7,
                            gbm_volatility=lambda jid, job: (float((jid % 21 - 10) * 1e-4), float((jid % 11) * 5e-3)))
    for jid in range(J):
        sw.add_metadata(jid, _Job(pb0, jid))
    sw.round_ptr = int(pb0["round_ptr"])

    def e2e_step():
        ids = sw.round_schedule()               # forced re-solve (resolve flag set below)
        for jid in ids[:G]:                     # what the round loop reports back (scheduler.py:2274-2341)
            job = sw.metadata[jid]
            sw.schedule_progress(jid, min(job.epochs, job.epoch_progress + (1 if jid % 3 == 0 else 0)))
        sw.increment_round_ptr()
        sw.set_resolve()
        return len(ids)

    for _ in range(W):
        e2e_step()
    if world > 1:
        dist.barrier()
    sampler.t1 = None
    t0 = time.perf_counter()
    for _ in range(K):
        e2e_step()
    e2e_s = time.perf_counter() - t0
    sampler.t1 = time.perf_counter()
    te = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_val = world * K / float(te.item())
    rs_kern = eng_t = sw._eng().last_timings()
    h2d = J * (4 + 4 + 8 + 4) + 256                      # slots, epoch_progress, measured samples, last round; params
    d2h = J * (16 * 2 + 4 + 6 * 8) + 64                  # two 128-bit masks/job, counts, six forecast planes; scalars
    # the same call without the Monte-Carlo stage, and its host part alone
    sw_det = ShockwaveScheduler(ngpus=G, gram=16, init_metadata=OrderedDict(), future_nrounds=T, round_duration=int(D),
                                solver_preference=["GUROBI"], solver_rel_gap=1e-3, solver_num_threads=24,
                                solver_timeout=15, n_epoch_vars_max=64, logapx_bases=BASES, logapx_origin=ORIGIN,
                                k=1e-3, lam=12.0, rhomax=1.0, device=local)
    for jid in range(J):
        sw_det.add_metadata(jid, _Job(pb0, jid))
    det_ms = []
    for i in range(W + 8):
        sw_det.round_ptr = int(pb0["round_ptr"]) + i
        sw_det.set_resolve()
        t0 = time.perf_counter()
        sw_det.round_schedule()
        det_ms.append((time.perf_counter() - t0) * 1e3)
    det_ms = float(np.median(det_ms[W:]))
    det_kern = sw_det._eng().last_timings()
    sampler.stop_flag = True
    del sw, sw_det

    extras = {}
    if not args.no_extras:
        extras = run_extras(args, eng, dev, dist, world, rank, local, est, flush, W, pbs)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    clocks = sampler.summary()
    ms_solve, ms_place = float(np.mean(ksolve)), float(np.mean(kplace))
    step_ms = total_ms / K
    line = {
        "metric": METRIC, "value": value, "unit": "rounds/s", "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64 (job scalars, objective, forecast sums); price thresholds compared in fp32; GBM paths in fp32",
        "data": "synthetic", "config": CONFIG,
        "timing": {"l2": "flushed between timed steps (256 MiB write)", "events": "CUDA events on the launching "
                   "stream around every step (forecast / ensemble / solve+place queued back to back, one synchronise at the end of the solve call), summed, max over ranks",
                   "numa_binding": numa},
        "clocks": clocks,
        "gpu_launches": gpu_launches,
        "step": {"fallback_steps": nfb, "unseated_job_rounds": shortf, "mc_paths_per_job": P_MC,
                 "kernels_ms": {"gbm_kernel": mc_ms, "solve_kernel": ms_solve, "place_kernel": ms_place},
                 "kernel_share_of_step": {"gbm_kernel": mc_ms / step_ms, "solve_kernel": ms_solve / step_ms,
                                          "place_kernel": ms_place / step_ms},
                 "bounds": {"gbm_kernel": "ALU/SFU (xorshift128+, Box-Muller, exp per path step)",
                            "solve_kernel": "instruction issue + barrier latency (8-CTA cluster, DSMEM reductions)",
                            "place_kernel": "latency (sorts, scans and the round packer in shared memory, one CTA)"}},
        "e2e": {"value": e2e_val, "unit": "rounds/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "what": "ShockwaveScheduler(forecast='gbm').round_schedule() with a forced re-solve per step, "
                        f"4096 live jobs, {G} schedule_progress() calls between steps (timed too)",
                "ms_per_call": 1e3 * float(te.item()) / K,
                "without_monte_carlo_ms_per_call": det_ms,
                "kernels_ms_without_monte_carlo": det_kern},
    }
    line.update(extras)
    if not args.no_cpu_baseline and world == 1:
        line["cpu_baseline"] = cpu_baseline_sample()
        line["same_algorithm_cpu"] = same_algorithm_cpu()
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def dump_outputs(out_dir, res, rem, xm, bm, nr):
    """The last timed step as a caller of it receives it: the Monte-Carlo mean remaining runtimes the solve planned with
    (remaining_runtime [J]), the round and back-fill schedules unpacked from their 128-bit masks (x, backfill [J, T]),
    the rounds per job (nrounds [J]) and the solve's result record (result: the swb_result fields in declaration order)."""
    from shockwave_b200.engine import Result, unpack_masks
    os.makedirs(out_dir, exist_ok=True)
    masks = lambda t: unpack_masks(t[0].cpu().numpy().view(np.uint64), T).astype(np.float32)
    arrays = {"remaining_runtime": rem[0].cpu().numpy().astype(np.float64), "x": masks(xm), "backfill": masks(bm),
              "nrounds": nr[0].cpu().numpy().astype(np.float32),
              "result": np.array([float(res[f]) for f, _ in Result._fields_], dtype=np.float64)}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def cpu_baseline_sample():
    """Bounded CPU sample (10-30 s): a full config-D MILP needs minutes of HiGHS (see --impl reference, which times it
    on the same seeds), so the sample is the largest BASELINE size the oracle finishes inside the budget — config C
    (1024 jobs x 128 GPUs x 32 rounds) — solved by the oracle with the reference's settings AND by the GPU path."""
    from oracle import shockwave_milp as om
    from shockwave_b200 import Engine, make_params
    from tests.synth import synth_problem
    logv = om.pwl_log_values(BASES, ORIGIN)
    Jc, Gc, Tc = 1024, 128, 32
    times, oks, gaps = [], 0, []
    eng = Engine(int(os.environ.get("LOCAL_RANK", "0")))
    gpu_ms = []
    for s in range(3):
        pb = synth_problem(Jc, Gc, Tc, D, seed=900 + s, tight=3.0)
        t0 = time.perf_counter()
        out = None
        try:
            out = om.dynamic_eisenberg_gale(pb["g"], pb["E"], pb["c"], pb["dbar"], pb["rem"], pb["ftobj"], Gc, Tc, D,
                                            pb["round_ptr"], 1e-3, 12.0, 1.0, BASES, logv, rel_gap=1e-3,
                                            time_limit=15.0, do_rank=False)
            om.construct_schedules(out["x"], list(range(Jc)), pb["g"], pb["rem"], pb["round_ptr"], Gc)
            oks += 1
        except AssertionError:
            pass
        times.append(time.perf_counter() - t0)
        prm = make_params(Gc, Tc, D, 1e-3, 12.0, 1.0, BASES, ORIGIN, round_ptr=pb["round_ptr"])
        for _ in range(3):
            t0 = time.perf_counter()
            o = eng.solve(prm, pb["g"], pb["E"], pb["c"], pb["dbar"], pb["rem"], pb["ftobj"], packed=True)
            g_ms = (time.perf_counter() - t0) * 1e3
        gpu_ms.append(g_ms)
        if out is not None:
            gaps.append((o["results"][0]["objective"] - out["objective"]) / abs(out["objective"]))
    val = len(times) / sum(times)
    return {"value": val, "unit": "rounds/s", "cores": 1, "kind": "port", "host_cores": os.cpu_count(),
            "workload": "BASELINE config C: 1024 jobs x 128 GPUs x 32-round window (NOT the headline size)",
            "gpu_same_instances_rounds_per_s": 1e3 / float(np.mean(gpu_ms)),
            "gpu_over_cpu_same_instances": (1e3 / float(np.mean(gpu_ms))) / val,
            "gpu_objective_minus_cpu_objective_rel": gaps,
            "sample": (f"3 config-C scenarios (seeds 900-902) through oracle/shockwave_milp.py (HiGHS, mip_rel_gap=1e-3, "
                       f"time_limit=15 s = the reference's settings) + construct_schedules, one core: {[round(t, 2) for t in times]} s, "
                       f"incumbents {oks}/3; the same three instances through Engine.solve with host buffers: "
                       f"{[round(m, 3) for m in gpu_ms]} ms; the headline size (config D) needs minutes per scenario on "
                       "one core — timed on the same seeds by `bench.py --impl reference`")}


def same_algorithm_cpu(nscn=None):
    """The SAME algorithm as solve.cu (collapsed MILP: clearing price nested in a makespan search) as plain C on ALL host
    cores, one config-D scenario per OpenMP thread (oracle/price_search.c) — separates what the algorithm buys from what
    the B200 buys.  Counts only (no placement / back-fill), float64."""
    from oracle import price_search as ps
    from oracle import shockwave_milp as om
    ncpu = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    S = nscn or max(8, min(2 * ncpu, 256))
    pbs = [scenario(i) for i in range(S)]
    st = lambda key: np.stack([p[0][key] for p in pbs])
    logv = om.pwl_log_values(BASES, ORIGIN)
    arrs = [st(k) for k in ("g", "E", "c", "dbar", "rem", "ftobj")]
    ks, rps = [p[1] for p in pbs], [p[0]["round_ptr"] for p in pbs]
    ps.price_search(ks[:ncpu], rps[:ncpu], *[a[:ncpu] for a in arrs], G, T, D, 12.0, 1.0, BASES, logv, ncpu)   # warm-up
    t0 = time.perf_counter()
    r = ps.price_search(ks, rps, *arrs, G, T, D, 12.0, 1.0, BASES, logv, ncpu)
    dt = time.perf_counter() - t0
    t0 = time.perf_counter()
    ps.price_search(ks[:4], rps[:4], *[a[:4] for a in arrs], G, T, D, 12.0, 1.0, BASES, logv, 1)
    one = (time.perf_counter() - t0) / 4
    return {"value": S / dt, "unit": "rounds/s", "threads": ncpu, "scenarios": S, "seconds_per_scenario_one_core": one,
            "mean_price_evaluations": float(np.mean(r["evals"])),
            "what": "oracle/price_search.c: the collapsed solve of solve.cu restated in plain C (float64, gcc -O3, OpenMP, "
                    "one scenario per thread), round counts only — no placement, back-fill or forecast"}


def run_extras(args, eng, dev, dist, world, rank, local, est, flush, W, pbs):
    """Legs that explain the headline: batched scenario sweep (+ path-sharded GBM with one all-reduce), the dense
    PR-dynamics pass (HBM roofline kernel, SURVEY.md §8d), single re-solve latency, Gavel get_allocation() latency."""
    import torch
    from shockwave_b200 import make_params
    from shockwave_b200.forecast_mc import path_range
    out = {}
    S, P_MC = args.scenarios, args.mc_paths
    # ONE job set shared by all ranks (the sweep forecasts it with paths sharded over the ranks): rank 0's scenario 0 —
    # `pbs` holds a different scenario stream per rank
    pb0 = scenario(0, 0)[0]
    # ---- batched: S what-if scenarios of ONE job set per step ------------------------------------------------
    rep = lambda a, dt: torch.from_numpy(np.ascontiguousarray(np.broadcast_to(a.astype(dt), (S, J)))).to(dev)
    bt = dict(g=rep(pb0["g"], np.int32), E=rep(pb0["E"], np.int32), c=rep(pb0["c"], np.int32),
              dbar=rep(pb0["dbar"], np.float64), ftobj=rep(pb0["ftobj"], np.float64))
    RH = [1.0, 1.5, 3.0, 10.0]
    zq = np.linspace(-1.5, 1.5, S)
    bprm = [make_params(G, T, D, K_SWEEP[s % 3], 12.0, RH[(s // 3) % 4], BASES, ORIGIN, round_ptr=pb0["round_ptr"])
            for s in range(S)]
    rem_s = torch.zeros((S, J), dtype=torch.float64, device=dev)
    R0 = torch.from_numpy(pb0["rem"]).to(dev)
    Hh = torch.from_numpy(np.minimum(pb0["E"] - pb0["c"], 256).astype(np.int32)).to(dev)
    rng = np.random.default_rng(99)
    mu = torch.from_numpy(rng.uniform(-1e-3, 1e-3, J)).to(dev)
    sg = torch.from_numpy(rng.uniform(0.0, 0.05, J)).to(dev)
    sums = torch.zeros((2, J), dtype=torch.float64, device=dev)
    bxm = torch.zeros((S, J, 2), dtype=torch.int64, device=dev)
    bbm = torch.zeros((S, J, 2), dtype=torch.int64, device=dev)
    lo, nloc = path_range(P_MC, rank, world)
    bptrs = {k: v.data_ptr() for k, v in bt.items()}
    bptrs["rem"] = rem_s.data_ptr(); bptrs["bfkey"] = rem_s.data_ptr()

    def bstep():
        eng.gbm_forecast_device(J, R0.data_ptr(), Hh.data_ptr(), mu.data_ptr(), sg.data_ptr(), nloc, lo, 11,
                                sums.data_ptr())
        if world > 1:
            dist.all_reduce(sums, op=dist.ReduceOp.SUM)        # NCCL over NVLink: [2][J] float64 = 64 KiB
            torch.cuda.current_stream(dev).synchronize()
        eng.gbm_ensemble(S, J, P_MC, sums.data_ptr(), zq, rem_s.data_ptr())
        return eng.solve_device(bprm, J, bptrs, dict(xmask=bxm.data_ptr(), bfmask=bbm.data_ptr()))

    for _ in range(3):
        res = bstep()
    if world > 1:
        # N > 1 correctness of the sharded forecast, checked by every driver run: the all-reduced sums must equal a
        # rank-0 recompute of ALL paths (path streams are keyed by the global path id)
        full = torch.zeros((2, J), dtype=torch.float64, device=dev)
        eng.gbm_forecast_device(J, R0.data_ptr(), Hh.data_ptr(), mu.data_ptr(), sg.data_ptr(), P_MC, 0, 11,
                                full.data_ptr())
        rel = float(((sums - full).abs() / full.abs().clamp_min(1e-300)).max().item())
        assert rel < 1e-9, f"sharded GBM forecast differs from the single-GPU recompute: {rel}"
        out["mc_shard_check_rel"] = rel
    KB = 5
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(KB)]
    ks, kp = [], []
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    for i in range(KB):
        flush.fill_(i)
        torch.cuda.synchronize()
        ev[i][0].record(est)
        res = bstep()
        ev[i][1].record(est)
        tm = eng.last_timings()
        ks.append(tm["ms_solve"]); kp.append(tm["ms_place"])
    torch.cuda.synchronize()
    bms = sum(a.elapsed_time(b) for a, b in ev)
    tb = torch.tensor([bms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tb, op=dist.ReduceOp.MAX)
    bms = float(tb.item())
    out["batched"] = {"value": world * S * KB / (bms * 1e-3), "unit": "rounds/s", "scenarios_per_gpu_per_step": S,
                      "steps": KB, "ms_per_step": bms / KB,
                      "what": "GBM forecast of one job set (paths sharded over the ranks, one NCCL all-reduce of 64 KiB) "
                              "-> S scenarios = k x rhomax x forecast quantile (z in [-1.5, 1.5]) -> solve + placement, "
                              "one CTA per scenario, packed round masks out; inputs resident",
                      "fallback_scenarios": sum(1 for r in res if r["status"] == 1),
                      "kernels_ms": {"solve_kernel": float(np.mean(ks)), "place_kernel": float(np.mean(kp))},
                      "mc_paths_this_rank": nloc}
    del bt, rem_s, bxm, bbm
    if rank != 0:
        return out

    # ---- single re-solve latency (S = 1, resident, no Monte-Carlo) -------------------------------------------
    dt1 = {k: torch.from_numpy(np.ascontiguousarray(pb0[k].astype(dtp))).to(dev)
           for k, dtp in (("g", np.int32), ("E", np.int32), ("c", np.int32), ("dbar", np.float64),
                          ("rem", np.float64), ("ftobj", np.float64))}
    xm1 = torch.zeros((1, J, 2), dtype=torch.int64, device=dev)
    bm1 = torch.zeros((1, J, 2), dtype=torch.int64, device=dev)
    lat = {}
    for name, cl in (("cluster8", 8), ("one_cta", 1)):
        eng.set_option(2, cl)
        ws = []
        for i in range(W + 8):
            t0 = time.perf_counter()
            eng.solve_device([make_params(G, T, D, 1e-3, 12.0, 1.0, BASES, ORIGIN, round_ptr=pb0["round_ptr"])], J,
                             {k: v.data_ptr() for k, v in dt1.items()}, dict(xmask=xm1.data_ptr(), bfmask=bm1.data_ptr()),
                             per_scenario_jobs=False)
            ws.append((time.perf_counter() - t0) * 1e3)
        lat[name] = {"wall_ms": float(np.median(ws[W:])), **eng.last_timings()}
    eng.set_option(2, 8)
    out["latency_S1"] = lat

    # ---- dense PR-dynamics pass over X[S][J][W][T] (SURVEY.md §8d): S*J*W*T*4 B = 512 MiB > L2 ------------------
    from shockwave_b200.engine import market_pgd
    Sd, Wd = 512, 1
    Xd = torch.zeros((Sd, J, Wd, T), dtype=torch.float32, device=dev)
    dj = {k: torch.from_numpy(np.ascontiguousarray(pb0[k]).astype(np.float64 if k != "g" else np.int32)).to(dev)
          for k in ("g", "E", "c", "dbar", "rem")}
    drate = torch.from_numpy((D / pb0["dbar"])[:, None].astype(np.float32)).to(dev)
    mptr = dict(shape=(Sd, J, Wd, T), per_scenario_jobs=0, g=dj["g"].data_ptr(), E=dj["E"].data_ptr(),
                c=dj["c"].data_ptr(), dbar=dj["dbar"].data_ptr(), rem=dj["rem"].data_ptr(), rate=drate.data_ptr(),
                X=Xd.data_ptr())
    mprm = [make_params(G, T, D, 1e-9, 12.0, 1.0, BASES, ORIGIN) for _ in range(Sd)]
    dense_ms = []
    for i in range(W + 5):
        # 150 passes on the time-coarsened tensor, then 16 full passes, each timed with its own event pair (ms = their
        # mean): the timed passes work on a converged, non-trivial allocation, not on zeros
        mobj, ms = market_pgd(eng, mprm, None, None, None, None, None, None, [G], None, 16, coarse_iters=150,
                              device_ptrs=mptr)
        if i >= W:
            dense_ms.append(ms)
    dense_ms = float(np.mean(dense_ms))
    # the same iteration as a SOLVER on one config-D scenario: objective of its feasible tensor against the exact optimum of
    # the same relaxation from the collapsed price search (solve.cu, itself pinned on the HiGHS LP in the tests)
    eng.set_option(1, 1)
    ex = eng.solve(make_params(G, T, D, 1e-9, 12.0, 1.0, BASES, ORIGIN, round_ptr=pb0["round_ptr"]), pb0["g"], pb0["E"],
                   pb0["c"], pb0["dbar"], pb0["rem"], 1e30 * np.ones(J))["results"][0]["relaxed_objective"]
    eng.set_option(1, 0)
    X1 = np.zeros((1, J, 1, T), dtype=np.float32)
    t0 = time.perf_counter()
    o1, _ = market_pgd(eng, mprm[0], pb0["g"], pb0["E"], pb0["c"], pb0["dbar"], pb0["rem"],
                       (D / pb0["dbar"])[:, None].astype(np.float32), [G], X1, 300, coarse_iters=1000)
    dense_solver = {"passes_full": 300, "passes_coarse": 1000, "objective": float(o1[0, 0]), "exact_relaxation": float(ex),
                    "relative_gap": float((ex - o1[0, 0]) / abs(ex)), "wall_ms_incl_copies": (time.perf_counter() - t0) * 1e3,
                    "what": "config D, W = 1, k = 1e-9 (welfare only): two-level PDHG from X = 0 vs the exact relaxed optimum"}
    dense_bytes = 8.0 * Sd * J * Wd * T + Sd * (24.0 * J + 8.0 * Wd * T)
    del Xd
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    traffic, trow = _ncu_traffic("market_step")
    out["roofline"] = {
        "bound": "hbm", "kernel": "market_step_fast<1,4,16> (dense PR-dynamics pass over X[S][J][W][T], fp32)",
        "achieved": dense_bytes / (dense_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
        "frac": dense_bytes / (dense_ms * 1e-3) / 1e9 / peak, "traffic": traffic,
        "traffic_source": "profiles/ncu_kernels_r02.json (ncu --set full of this command)" if traffic else None,
        "algorithmic_bytes_per_launch": dense_bytes, "shape": [Sd, J, Wd, T], "ms_per_launch": dense_ms,
        "as_solver": dense_solver,
        "note": "the kernel SURVEY.md §8(d) designates for the HBM roofline; algorithmic bytes = 8*S*J*W*T + "
                "S*(24*J + 8*W*T); tensor (512 MiB) larger than L2; timed live with CUDA events on the launching stream "
                "around each of the 16 full dense passes of a run of 150 coarse + 16 full PDHG iterations (mean of 16 x 5 launches), in its own leg: the kernels of the timed step (`step`) are "
                "ALU- and latency-bound, never HBM-bound, and are listed with those bounds; peak = MEASURED_PEAKS.json "
                "hbm_gbs" + ("" if peaks else " (fallback 6650)")}

    # ---- config E (J=2048 policy sweep): Gavel get_allocation() latency, W=1 (pooled) and W=3 (heterogeneous) ----
    from shockwave_b200 import policies as GP
    GP._shared_engine = eng
    rngp = np.random.default_rng(7)
    JE = 2048
    mE = rngp.uniform(0.5, 20.0, size=(JE, 1)) * np.sort(rngp.uniform(0.1, 1.0, size=(JE, 3)), axis=1)
    wts = ["k80", "p100", "v100"]
    thr3 = {j: {w: float(mE[j, i]) for i, w in enumerate(wts)} for j in range(JE)}
    thr1 = {j: {w: float(mE[j, 2]) for w in wts} for j in range(JE)}
    sfE = {j: int(rngp.choice([1, 2, 4, 8], p=[0.6, 0.3, 0.09, 0.01])) for j in range(JE)}
    prE = {j: 1.0 for j in range(JE)}
    stE = {j: float(rngp.uniform(1e4, 1e6)) for j in range(JE)}
    tE = {j: float(rngp.uniform(0, 5e3)) for j in range(JE)}
    pol_ms = {}
    for tag, thr_, spec_ in (("W1", thr1, {"k80": 0, "p100": 0, "v100": 512}),
                             ("W3", thr3, {"k80": 256, "p100": 128, "v100": 128})):
        for name, call in (
                ("max_min_fairness_perf", lambda: GP.MaxMinFairnessPolicyWithPerf("ECOS").get_allocation(thr_, sfE, prE, spec_)),
                ("finish_time_fairness_perf", lambda: GP.FinishTimeFairnessPolicyWithPerf("GUROBI").get_allocation(
                    thr_, sfE, prE, tE, stE, spec_)),
                ("max_min_fairness_water_filling_perf", lambda: GP.MaxMinFairnessWaterFillingPolicyWithPerf().get_allocation(
                    thr_, sfE, prE, spec_))):
            call()
            t0 = time.perf_counter()
            for _ in range(3):
                call()
            pol_ms[f"{name}_{tag}"] = (time.perf_counter() - t0) / 3 * 1e3
    out["gavel_get_allocation_ms_J2048"] = pol_ms

    # ---- packing policies (space sharing): LPs over (job combination x worker type) columns on swb_lp_solve ----
    try:
        out["packed_get_allocation_ms"] = bench_packed(GP)
    except Exception as e:            # an auxiliary leg: never take the headline down with it
        out["packed_get_allocation_ms"] = {"error": repr(e)}

    # ---- simulator round loop (SURVEY 8f-4): what-if replays of the reference's recorded 643-round schedule ----
    try:
        out["sim_round_loop"] = bench_sim_loop(local)
    except Exception as e:            # an auxiliary leg: never take the headline down with it
        out["sim_round_loop"] = {"error": repr(e)}
    return out


def bench_packed(GP):
    from shockwave_b200 import packing as PK
    from tests.packing_fixtures import instance as packed_instance
    pk_ms = {}
    for ns in (32, 64):
        thr_p, sf_p, pr_p, t_p, st_p, spec_p, _ = packed_instance(ns, {"v100": 16, "p100": 12, "k80": 8}, seed=ns)
        for name, call in (
                ("max_min_fairness_packed", lambda: GP.get_policy("max_min_fairness_packed", "ECOS").get_allocation(
                    thr_p, sf_p, pr_p, spec_p)),
                ("finish_time_fairness_packed", lambda: GP.get_policy("finish_time_fairness_packed", "ECOS").get_allocation(
                    thr_p, sf_p, pr_p, t_p, st_p, spec_p))):
            call()
            t0 = time.perf_counter()
            for _ in range(3):
                call()
            pk_ms[f"{name}_{ns}jobs_{len(thr_p)}combinations"] = (time.perf_counter() - t0) / 3 * 1e3
        stats = getattr(getattr(PK, "_max_min", None), "last_stats", None)
        if stats is not None:
            pk_ms[f"simplex_pivots_{ns}jobs"] = int(np.asarray(stats)[:, 0].max())
    return pk_ms


def bench_policy_ensemble(device):
    """8 what-ifs of the canonical 120-job trace AS SHIPPED (accordion / gns jobs) under max-min fairness on 32 GPUs:
    allocation kernels + swb_gavel_round + the device round loop, no reference code in the loop.  The reference's own run
    of this policy on this trace is on record (tests/golden/sim_dynamic_pins.json, unmodified simulator): the makespan and
    every completion time must come out the same."""
    from shockwave_b200 import policies as GP
    from shockwave_b200.simulate import PolicyEnsemble
    d = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "tests", "golden", "sim_dynamic_pins.json")))
    rec, dyn = d["max_min_fairness_32"], d["fifo_32"]["dyn"]
    tr = {k: np.asarray(rec[k]) for k in ("arrival", "total_steps", "scale_factor", "throughput", "duration", "batch_size",
                                          "dataset_len")}
    S = 8
    ens = PolicyEnsemble(tr, [GP.get_policy("max_min_fairness", solver="ECOS", seed=0) for _ in range(S)], rec["ngpus"],
                         time_per_iteration=rec["time_per_iteration"], device=device, dynamic=dyn)
    t0 = time.perf_counter()
    out = ens.run()
    dt = time.perf_counter() - t0
    J = len(rec["arrival"])
    want = np.array([rec["jct"][str(j)] for j in range(J)])
    return {"what": "PolicyEnsemble: max_min_fairness, canonical trace as shipped, 32 GPUs", "scenarios": S,
            "rounds": int(out["rounds"][0]), "seconds": dt, "seconds_per_scenario": dt / S,
            "allocations_per_scenario": int(out["allocations"][0]),
            "makespan": float(out["makespan"][0]), "reference_makespan": rec["makespan"],
            "jobs_with_identical_completion_time": int((out["jct"][S - 1] == want).sum()), "jobs": J,
            "max_rel_completion_time_difference": float(np.max(np.abs(out["jct"][S - 1] / want - 1.0))),
            "note": "the recorded run used the HiGHS-backed policy code (build container); the device policy returns the "
                    "same optimal value and its own point of the optimal face, so single completion times may move",
            "reference_loop_seconds_note": "1.5-2.1 s per run of the unmodified loop with the same device policies "
                                           "(profiles/sim_ensemble_r02.json)"}


def bench_sim_loop(device):
    """S scenarios x R rounds of the static 120-job trace in ONE swb_sim_replay launch (the schedule the unmodified
    reference recorded under max_min_fairness on 12 GPUs, tests/golden/sim_static_pins.json), checked against the
    recorded completion times; beside it the pinned restatement (oracle/sim_loop.py, one core) on the same schedule."""
    from shockwave_b200.simulate import DeviceSim
    rec = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "tests", "golden",
                                      "sim_static_pins.json")))["max_min_fairness_12"]
    tr = {k: np.asarray(rec[k]) for k in ("arrival", "total_steps", "scale_factor", "throughput", "duration", "batch_size",
                                          "dataset_len")}
    J, R = len(rec["arrival"]), len(rec["per_round_schedule"])
    mask = np.zeros((R, J), np.uint8)
    for r, ids in enumerate(rec["per_round_schedule"]):
        mask[r, ids] = 1
    S = 148 * 8
    sim = DeviceSim(tr, S, rec["ngpus"], rec["time_per_iteration"], device=device)
    sim.replay(mask)                                   # warm-up (+ first-touch of the arena)
    t0 = time.perf_counter()
    reps = 5
    for _ in range(reps):
        scn = sim.replay(mask)
    dt = (time.perf_counter() - t0) / reps
    res = sim.results()
    want = np.array([rec["jct"][str(j)] for j in range(J)])
    ok = bool(np.array_equal(res["jct"][0], want) and np.array_equal(res["jct"][S - 1], want) and
              (scn["rounds"] == rec["rounds"]).all())
    sim.close()
    from oracle import sim_loop                      # CPU leg only: the restatement as the one-core baseline
    t0 = time.perf_counter()
    sched = rec["per_round_schedule"]
    ora = sim_loop.run(rec, lambda c, now, active: sched[c], tpi=rec["time_per_iteration"])
    t_cpu = time.perf_counter() - t0
    ens = {}
    try:
        ens = bench_policy_ensemble(device)
    except Exception as e:
        ens = {"error": repr(e)}
    return {"policy_ensemble": ens,
            "what": "swb_sim_replay: begin + all rounds of S what-if scenarios in one launch, wall time incl. the H2D of "
                    "the schedule and the D2H of the scenario records",
            "scenarios": S, "rounds": R, "jobs": J, "ms_per_replay": dt * 1e3,
            "scenario_rounds_per_s": S * R / dt, "bit_identical_to_reference_records": ok,
            "cpu_restatement_rounds_per_s_one_core": R / t_cpu,
            "cpu_restatement_identical": bool(ora["makespan"] == rec["makespan"]),
            "reference_loop_note": "the unmodified reference loop itself: 303 rounds in 2.8 s with a solver-free policy "
                                   "(tests/golden/make_sim_pins.py, build container)"}


if __name__ == "__main__":
    main()
