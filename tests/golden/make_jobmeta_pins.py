"""Generator of tests/golden/jobmeta_pins.json.gz: the reference's own JobMetaData (scheduler/JobMetaData.py) on 40 random
job histories (tests/test_oracle_jobmeta.py::test_direct_against_reference_jobmetadata).  Recorded per job: what the
constructor derives from the profile (nworkers, epoch_duration_preprofiled, bs_schedule) and, after every step of the
history, the elapsed time, dirichlet_posterior_remaining_runtime() and the interpolated epoch duration.

    python -m tests.golden.make_jobmeta_pins         (needs the reference's scheduler/ directory, see oracle/ref_harness.py)
"""
import gzip
import json
import os
import sys
from collections import OrderedDict

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
PATH = os.path.join(ROOT, "tests", "golden", "jobmeta_pins.json.gz")


def histories():
    """(trial, profile, steps) of the 40 random jobs; steps = [(epoch progress, (round, (throughput, bs)) or None)]."""
    rng = np.random.default_rng(0)
    for trial in range(40):
        E = int(rng.integers(3, 60))
        nm = int(rng.integers(1, 4))
        modes = rng.choice([16, 32, 64, 128, 256], size=nm, replace=False)
        bs = np.sort(rng.choice(modes, size=E))
        dur = rng.uniform(5, 400, size=E)
        prof = dict(model="ResNet-18", dataset="CIFAR-10", num_samples_per_epoch=50000, num_epochs=E,
                    util_every_epoch=[1.0] * E, mem_every_epoch=[1000.0] * E,
                    duration_every_epoch=dur.tolist(), scale_factor=int(rng.choice([1, 2, 4])),
                    bs_every_epoch=[int(b) for b in bs])
        steps, rnd = [], 0
        for step in range(12):
            c = int(rng.integers(0, E + 1))
            entry = None
            if rng.random() < 0.7:
                rnd += int(rng.integers(1, 4))
                entry = (rnd, (float(rng.uniform(0.2, 30.0)), int(rng.choice(modes))))
            steps.append((c, entry))
        yield trial, prof, steps


def load():
    with gzip.open(PATH, "rt") as f:
        return json.load(f)


def main():
    sys.path.insert(0, ROOT)
    from oracle import ref_harness as rh
    sys.path.insert(0, rh.REF)
    from JobMetaData import JobMetaData
    out = []
    for trial, prof, steps in histories():
        ref = JobMetaData(trial, prof)
        tl = OrderedDict()
        ref.register_job_submit(123.0)
        ref.set_throughput_measurments(tl, 120)
        rec = dict(nworkers=int(ref.nworkers), pre=[float(v) for v in ref.epoch_duration_preprofiled],
                   bs=[int(v) for v in ref.bs_schedule], values=[])
        for c, entry in steps:
            ref.set_epoch_progress(c)
            if entry is not None:
                tl[entry[0]] = entry[1]
            ref.calibrate_profiled_epoch_duration()
            elapsed = float(sum(ref.epoch_duration[:c]))
            remaining = float(ref.dirichlet_posterior_remaining_runtime())
            ref.calibrate_profiled_epoch_duration()
            rec["values"].append([elapsed, remaining, float(np.mean(ref.epoch_duration[: c + 1]))])
        out.append(rec)
    with gzip.GzipFile(PATH, "wb", mtime=0) as f:
        f.write(json.dumps(out, separators=(",", ":")).encode())


if __name__ == "__main__":
    main()
