"""TEST INFRASTRUCTURE: build the UNMODIFIED reference simulator into oracle/_ref/ for the closed-loop tests.

The closed-loop parity tests (tests/test_closed_loop.py: the reference's own `Scheduler.simulate()` driving libswb200
through the drop-in classes, and the other tests that use oracle/ref_harness.py) need the reference's simulator next to a
B200.  When the reference's `scheduler/` directory is present at build time, this recipe byte-compiles its python files
(`scheduler/*.py`, `policies/`, `runtime/`) into sourceless `.pyc` modules under `oracle/_ref/scheduler/` and copies
the data the runs read: `configurations/`, `tacc_throughputs.json` / `wisr_throughputs.json`, the canonical 120-job
trace, the 220 / 460 / 900-job traces of `reproduce/scale_*gpus.sh` and the golden result pickles of
`reproduce/tacc_32gpus.sh` (about 8 MB).  `oracle/_ref/` is git-ignored: no reference source enters the repository.
Python imports the `.pyc` modules directly (sourceless loading), so the build is tied to the interpreter version that
made it.

Usage:  python -m oracle.stage_ref [--force]   (idempotent; run by __graft_entry__.build() when the reference exists)
"""
import os
import py_compile
import shutil
import sys
import warnings

SRC = "/root/reference/scheduler"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DST = os.path.join(ROOT, "oracle", "_ref", "scheduler")
TRACE = "traces/reproduce/120_0.2_5_100_40_25_0,0.5,0.5_0.6,0.3,0.09,0.01_multigpu_dynamic.trace"
# the 220-job trace of reproduce/scale_64gpus.sh (64 GPUs, wisr_throughputs.json) for the second closed-loop case
TRACE64 = "traces/reproduce/220_0.2_5_100_25_4_0,0.5,0.5_0.6,0.3,0.09,0.01_multigpu_dynamic.trace"
TRACE128 = "traces/reproduce/460_0.2_5_100_10_1_0,0.5,0.5_0.6,0.3,0.09,0.01_multigpu_dynamic.trace"
TRACE256 = "traces/reproduce/900_0.2_5_1000_5_15_0,0.5,0.5_0.6,0.3,0.09,0.01_multigpu_dynamic.trace"
SKIP = {"traces", "reproduce", "scripts", "__pycache__"}


def _build_tree(src, dst):
    for d, dirs, files in os.walk(src):
        dirs[:] = sorted(x for x in dirs if x not in SKIP)
        out = os.path.join(dst, os.path.relpath(d, src))
        os.makedirs(out, exist_ok=True)
        for f in files:
            if f.endswith(".png") or f == "actual_throughputs.json":
                continue
            if f.endswith(".py"):
                with warnings.catch_warnings():         # the reference's regex literals: SyntaxWarning, not ours to fix
                    warnings.simplefilter("ignore", SyntaxWarning)
                    py_compile.compile(os.path.join(d, f), cfile=os.path.join(out, f[:-3] + ".pyc"), doraise=True,
                                       dfile=os.path.join("scheduler", os.path.relpath(os.path.join(d, f), src)))
            else:
                shutil.copy(os.path.join(d, f), os.path.join(out, f))


def stage(force=False):
    if not os.path.isdir(SRC):
        return None
    if os.path.isdir(DST) and not force and os.path.exists(os.path.join(DST, TRACE256)):
        return DST
    if os.path.isdir(DST):
        shutil.rmtree(DST)
    _build_tree(SRC, DST)
    for t in (TRACE, TRACE64, TRACE128, TRACE256):
        os.makedirs(os.path.join(DST, os.path.dirname(t)), exist_ok=True)
        shutil.copy(os.path.join(SRC, t), os.path.join(DST, t))
    shutil.copytree(os.path.join(SRC, "reproduce", "pickles", "tacc_32gpus"),
                    os.path.join(DST, "reproduce", "pickles", "tacc_32gpus"))
    return DST


if __name__ == "__main__":
    print(stage(force="--force" in sys.argv))
