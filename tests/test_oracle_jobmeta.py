"""The numpy restatement of the forecast (oracle/jobmeta.py) against the reference's own JobMetaData:
 (a) through the committed fixture — values the reference objects produced inside the canonical
     simulation, replayed solve by solve (stateful calibration + share series included);
 (b) directly, on random job histories, against the values the reference's JobMetaData computed for them."""
import numpy as np
import pytest

from oracle import jobmeta as ojm
from tests import fixtures as fx
from tests.replay import replay_with_oracle_jobmeta


def test_replay_matches_reference_recorded_forecast():
    worst = dict(dbar=0.0, rem=0.0, ftobj=0.0)
    nbad = 0
    for i, s, out in replay_with_oracle_jobmeta():
        for key in ("dbar", "rem", "ftobj"):
            rel = np.abs(out[key] - s[key]) / np.maximum(1e-300, np.abs(s[key]))
            nbad += int(np.sum(rel > 1e-9))
            worst[key] = max(worst[key], float(rel.max()))
        if s["status"] == 1:
            rel = np.abs(out["rem_fb"] - s["rem_fb"]) / np.maximum(1e-300, np.abs(s["rem_fb"]))
            assert rel.max() <= 1e-9
    print("worst relative deviation", worst, "entries beyond 1e-9:", nbad)
    # float64 everywhere; only summation order differs from the reference (amp*sum vs sum(amp*x))
    assert worst["dbar"] <= 1e-9 and worst["rem"] <= 1e-9 and worst["ftobj"] <= 1e-9


def test_direct_against_reference_jobmetadata():
    """The restatement on 40 random job histories against what the reference's JobMetaData computed on the same
    histories (tests/golden/make_jobmeta_pins.py)."""
    from collections import OrderedDict
    from tests.golden import make_jobmeta_pins as pins
    recs = pins.load()
    for (trial, prof, steps), rec in zip(pins.histories(), recs):
        E = prof["num_epochs"]
        tl = OrderedDict()
        mine = ojm.JobState(trial, rec["nworkers"], E, 50000, rec["pre"], rec["bs"], 123.0, 120)
        mine.timeline = tl
        for (c, entry), (elapsed, remaining, interp) in zip(steps, rec["values"]):
            mine.epoch_progress = c
            if entry is not None:
                tl[entry[0]] = entry[1]
            mine.calibrate()
            assert np.isclose(mine.elapsed(), elapsed, rtol=1e-12)
            b = mine.remaining()
            assert np.isclose(remaining, b, rtol=1e-12), (trial, c, remaining, b)
            assert np.isclose(interp, mine.interpolate_epoch_duration(), rtol=1e-12)
    assert len(recs) == 40
