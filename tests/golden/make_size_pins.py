"""Generator of tests/golden/config_c_oracle.json and tests/golden/config_d_lp.json (BASELINE config C / D sizes).

Run here (no GPU, no reference needed; HiGHS through scipy):
    python tests/golden/make_size_pins.py c        # ~1 min   : MILP oracle at 1024 jobs x 128 GPUs (gap 1e-4)
    python tests/golden/make_size_pins.py d        # ~4 min   : LP relaxation at 4096 jobs x 512 GPUs x 64 rounds
    python tests/golden/make_size_pins.py d-milp   # ~10 min  : the MILP itself at config D with a 900 s limit (HiGHS needs
                                                   #            ~140 s per instance on one core; the reference's 15 s limit
                                                   #            yields no incumbent) -> config_d_milp.json
    python tests/golden/make_size_pins.py e        # ~18 min  : LP relaxation above 4096 jobs / 64 rounds -> limits_lp.json
                                                   #            (6144x768x64: 384 s, 8192x1024x32: 158 s, 5000x512x128:
                                                   #            498 s, one core each)
Inputs are tests/synth.py instances addressed by (J, G, T, seed, tight); the records keep those keys, the oracle's verdict
and objective and the seconds it took, so tests/test_gpu_solve.py can rebuild the instance and compare."""
import json
import os
import sys
import time

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from oracle import shockwave_milp as om          # noqa: E402
from tests.synth import synth_problem            # noqa: E402

BASES, ORIGIN = [0.0, 0.2, 0.4, 0.6, 0.8, 1.0], {0.0: 1e-6}
LOGV = om.pwl_log_values(BASES, ORIGIN)
D, LAM = 120.0, 12.0

CONFIG_C = [(1024, 128, 32, 1e-3, 1.0, 900), (1024, 128, 20, 1e-3, 3.0, 901), (1024, 128, 32, 1e1, 0.5, 902)]
CONFIG_D = [(4096, 512, 64, 1e-3, 3.0, 1000), (4096, 512, 64, 1e1, 3.0, 1001), (4096, 512, 64, 1e-3, 0.5, 1002)]
# the solve's global-memory path (J > 4096) and the high word of the 128-bit round masks (T > 64)
LIMITS = [(6144, 768, 64, 1e-3, 3.0, 1100), (8192, 1024, 32, 1e1, 3.0, 1101), (5000, 512, 128, 1e-3, 0.5, 1102)]


def milp(J, G, T, k, tight, seed, gap, limit):
    pb = synth_problem(J, G, T, D, seed=seed, tight=tight)
    t0 = time.time()
    out = om.dynamic_eisenberg_gale(pb["g"], pb["E"], pb["c"], pb["dbar"], pb["rem"], pb["ftobj"], G, T, D,
                                    pb["round_ptr"], k, LAM, 1.0, BASES, LOGV, rel_gap=gap, time_limit=limit,
                                    do_rank=False)
    return dict(J=J, G=G, T=T, k=k, tight=tight, seed=seed, D=D, lam=LAM, status=int(out["status"]),
                objective=float(out["objective"]), seconds=time.time() - t0)


def lp(J, G, T, k, tight, seed):
    pb = synth_problem(J, G, T, D, seed=seed, tight=tight)
    t0 = time.time()
    cap = om.ftf_caps(pb["rem"], pb["ftobj"], G, J, T, D, pb["round_ptr"], 1.0)
    status, w = om.STATUS_FTF_FEASIBLE, np.ones(J)
    ok, _, _, obj = om._solve(pb["g"].astype(np.int64), pb["E"].astype(float), pb["c"].astype(float), pb["dbar"],
                              pb["rem"], w, G, T, D, k, BASES, LOGV, cap, 1e-9, 0.0, relax=True)
    if not ok:
        status = om.STATUS_FALLBACK
        w, _ = om.relax_priorities(pb["rem"], pb["ftobj"], G, J, D, pb["round_ptr"], 1.0, LAM)
        ok, _, _, obj = om._solve(pb["g"].astype(np.int64), pb["E"].astype(float), pb["c"].astype(float), pb["dbar"],
                                  pb["rem"], w, G, T, D, k, BASES, LOGV, None, 1e-9, 0.0, relax=True)
    assert ok
    return dict(J=J, G=G, T=T, k=k, tight=tight, seed=seed, D=D, lam=LAM, status=int(status), lp_objective=float(obj),
                seconds=time.time() - t0)


if __name__ == "__main__":
    what = sys.argv[1] if len(sys.argv) > 1 else "c"
    if what == "c":
        recs = [milp(*p, gap=1e-4, limit=120.0) for p in CONFIG_C]
        path = "config_c_oracle.json"
    elif what == "d":
        recs = [lp(*p) for p in CONFIG_D]
        path = "config_d_lp.json"
    elif what == "e":
        recs = [lp(*p) for p in LIMITS]
        path = "limits_lp.json"
    else:
        recs = [milp(*p, gap=1e-3, limit=900.0) for p in CONFIG_D[:1]]
        path = "config_d_milp.json"
    for r in recs:
        print(r)
    json.dump(recs, open(os.path.join(HERE, path), "w"), indent=1)
