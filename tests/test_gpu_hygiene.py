"""Robustness of the C-ABI (round-1 review): gang widths are validated instead of truncated to a byte, the profile
pools of the resident job table do not grow with the number of jobs ever submitted, occupied slots are refused, and a
gang wider than the cluster gives the fallback verdict the reference's infeasible MILP gives."""
import numpy as np
import pytest

from oracle import shockwave_milp as om
from shockwave_b200 import make_params
from tests import fixtures as fx
from tests.synth import synth_problem

pytestmark = pytest.mark.gpu
LOGV = om.pwl_log_values(fx.BASES, fx.ORIGIN)


def _prm(G, T, r=0):
    return make_params(G, T, 120.0, 1e-3, 12.0, 1.0, fx.BASES, fx.ORIGIN, round_ptr=r)


@pytest.mark.parametrize("bad", [0, -3, 256, 300])
def test_solve_rejects_widths_outside_a_byte(engine, bad):
    pb = synth_problem(24, 512, 8, 120.0, seed=1)
    g = pb["g"].copy()
    g[5] = bad
    with pytest.raises(RuntimeError, match="gang width"):
        engine.solve(_prm(512, 8, pb["round_ptr"]), g, pb["E"], pb["c"], pb["dbar"], pb["rem"], pb["ftobj"])
    # and the context is still usable
    out = engine.solve(_prm(512, 8, pb["round_ptr"]), pb["g"], pb["E"], pb["c"], pb["dbar"], pb["rem"], pb["ftobj"])
    assert out["results"][0]["flags"] == 0


def test_device_resident_bad_width_is_reported(engine):
    import torch
    pb = synth_problem(24, 512, 8, 120.0, seed=2)
    g = pb["g"].copy()
    g[3] = 256                       # would truncate to 0 in a byte
    dev = torch.device("cuda", 0)
    t = {k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in
         dict(g=g.astype(np.int32), E=pb["E"].astype(np.int32), c=pb["c"].astype(np.int32), dbar=pb["dbar"],
              rem=pb["rem"], ftobj=pb["ftobj"]).items()}
    x = torch.zeros((1, 24, 8), dtype=torch.uint8, device=dev)
    with pytest.raises(RuntimeError, match="gang width"):
        engine.solve_device([_prm(512, 8)], 24, {k: v.data_ptr() for k, v in t.items()}, dict(x=x.data_ptr()))


def test_gang_wider_than_the_cluster_gives_the_reference_verdict(engine):
    """x_j = 0 is forced for g_j > G (capacity rows, shockwave.py:317); if that job's finish-time row needs rounds the
    reference MILP is infeasible and takes the fallback path — so must the kernel (it used to report OK)."""
    G, T, D = 8, 10, 120.0
    pb = synth_problem(12, G, T, D, seed=5, tight=3.0)
    g = pb["g"].copy(); g[:] = np.minimum(g, G); g[2] = 2 * G
    ftobj = pb["ftobj"].copy()
    ftobj[:] = 1e9                   # everybody else's row is slack ...
    ftobj[2] = D * (pb["round_ptr"] + T) + 10.0   # ... job 2 would need nearly all of its remaining runtime served
    ora = om.dynamic_eisenberg_gale(g, pb["E"], pb["c"], pb["dbar"], pb["rem"], ftobj, G, T, D, pb["round_ptr"],
                                    1e-3, 12.0, 1.0, fx.BASES, LOGV, rel_gap=1e-6, do_rank=False)
    out = engine.solve(_prm(G, T, pb["round_ptr"]), g, pb["E"], pb["c"], pb["dbar"], pb["rem"], ftobj)
    assert ora["status"] == om.STATUS_FALLBACK
    assert out["results"][0]["status"] == ora["status"]
    assert out["x"][0][2].sum() == 0


def test_profile_pool_tracks_live_jobs_not_history(engine):
    rng = np.random.default_rng(0)
    base = engine.job_table_stats()["used_rows"]
    slots = list(range(900, 916))
    E0 = [int(rng.integers(20, 200)) for _ in slots]
    for s, E in zip(slots, E0):
        engine.job_add(s, 1, E, 5e4, 0.0, rng.uniform(50, 500, E), np.full(E, 32))
    live = engine.job_table_stats()["used_rows"] - base
    assert live == sum(E + 1 for E in E0)
    with pytest.raises(RuntimeError, match="occupied"):
        engine.job_add(slots[0], 1, 10, 5e4, 0.0, np.ones(10), np.full(10, 32))
    # churn: 400 generations of remove + add of jobs no larger than the ones they replace
    for gen in range(400):
        k = int(rng.integers(0, len(slots)))
        engine.job_remove(slots[k])
        E = int(rng.integers(10, E0[k] + 1))
        engine.job_add(slots[k], 1, E, 5e4, 0.0, rng.uniform(50, 500, E), np.full(E, 32))
    st = engine.job_table_stats()
    assert st["used_rows"] - base <= live, st       # round 1: grew by every job ever added
    for s in slots:
        engine.job_remove(s)
    assert engine.job_table_stats()["used_rows"] == base


@pytest.mark.parametrize("J,G,T,k", [(512, 128, 32, 1e-3), (1000, 128, 20, 1e1), (4096, 512, 64, 1e-3),
                                     (4096, 512, 64, 1e5), (3000, 96, 64, 1e1)])
def test_cluster_solve_equals_single_cta_solve(engine, J, G, T, k):
    """Latency path: a cluster of 8 CTAs shares one scenario (DSMEM reductions in rank order).  Same searches on the
    same step functions -> the same round counts as the one-CTA kernel; the objective may differ in the last bits
    (summation order)."""
    engine.set_option(6, 0)        # re-rank search off: with it the cluster size also selects single / multi-start placement
    for seed, tight in ((0, 3.0), (1, 0.5)):
        pb = synth_problem(J, G, T, 120.0, seed=seed, tight=tight)
        prm = make_params(G, T, 120.0, k, 12.0, 1.0, fx.BASES, fx.ORIGIN, round_ptr=pb["round_ptr"])
        outs = []
        for cl in (1, 8):
            engine.set_option(2, cl)       # SWB_OPT_SOLVE_CLUSTER
            outs.append(engine.solve(prm, pb["g"], pb["E"], pb["c"], pb["dbar"], pb["rem"], pb["ftobj"]))
        engine.set_option(2, 8)
        a, b = outs
        assert a["results"][0]["status"] == b["results"][0]["status"]
        assert np.array_equal(a["nrounds"], b["nrounds"])
        assert np.array_equal(a["x"], b["x"])
        assert abs(a["results"][0]["objective"] - b["results"][0]["objective"]) <= 1e-9 * abs(a["results"][0]["objective"])
    engine.set_option(6, 400)


def test_solve_cluster_option_belongs_to_its_engine(engine):
    """SWB_OPT_SOLVE_CLUSTER = 1 on one Engine leaves another Engine's fallback placement on its 8-start re-rank search
    (thread-block cluster): a recorded canonical fallback solve whose best start is not start 0 (flags >> 20) gives the
    same schedule and flags before and after the option is set elsewhere."""
    from shockwave_b200 import Engine
    T, G, D = fx.TACC["T"], fx.TACC["G"], fx.TACC["D"]

    def run(s):
        prm = make_params(G, T, D, fx.TACC["k"], fx.TACC["lam"], fx.TACC["rhomax"], fx.BASES, fx.ORIGIN,
                          round_ptr=s["round_ptr"])
        return engine.solve(prm, s["g"], s["E"], s["c"], s["dbar"], s["rem"], s["ftobj"], bfkey=s["rem"])

    cases = []
    for i in range(fx.n_solves()):
        s = fx.solve(i)
        if s["status"] == om.STATUS_FALLBACK:
            out = run(s)
            if out["results"][0]["flags"] >> 20:
                cases.append((s, out))
    assert cases, "no recorded fallback solve is won by a noised start"
    other = Engine(0)
    try:
        other.set_option(2, 1)
        for s, before in cases[:8]:
            after = run(s)
            assert after["results"][0]["flags"] == before["results"][0]["flags"]
            assert np.array_equal(after["x"], before["x"])
    finally:
        other.close()
