"""CPU tests: the C-ABI library loads and exports every symbol include/swb200.h declares (no compute
without a GPU), struct layouts agree, and the host state machine of the drop-in class."""
import ctypes as C
import os
import re
import shutil
import subprocess
from collections import OrderedDict

import numpy as np
import pytest

from shockwave_b200 import engine
from shockwave_b200.scheduler import ShockwaveScheduler, schedules_from_matrices

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header_text():
    txt = open(os.path.join(ROOT, "include", "swb200.h")).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return re.sub(r"^\s*#.*$", "", txt, flags=re.M)


def _header_functions():
    return sorted(set(re.findall(r"\b(swb_[a-z_0-9]+)\s*\(", _header_text())))


def _header_prototypes():
    """{name: (return type, [parameter types])} of every function the header declares."""
    protos = {}
    for ret, name, params in re.findall(r"(?:^|(?<=[;{}]))\s*([^;{}()]*?)\b(swb_[a-z_0-9]+)\s*\(([^()]*)\)\s*;",
                                        _header_text()):
        params = [p.strip() for p in params.split(",")]
        if params == ["void"]:
            params = []
        # drop the parameter name: what is left is its type
        protos[name] = (ret.strip(), [re.sub(r"\b[A-Za-z_]\w*$", "", p).strip() or p for p in params])
    return protos


def _c_kind(ctype):
    if "*" in ctype:
        return "ptr"
    base = ctype.replace("const", "").strip()
    return {"void": "void", "int": "i32", "int32_t": "i32", "int64_t": "i64", "uint64_t": "u64",
            "double": "f64", "float": "f32"}[base]


def _ctypes_kind(t):
    if t is None:
        return "void"
    if issubclass(t, C._Pointer):
        return "ptr"
    code = {"P": "ptr", "z": "ptr", "d": "f64", "f": "f32"}.get(t._type_)
    if code:
        return code
    signed = t._type_.islower()
    return {4: "i32" if signed else "u32", 8: "i64" if signed else "u64"}[C.sizeof(t)]


def test_library_exports_every_declared_symbol():
    lib = engine.load_library()
    names = _header_functions()
    assert len(names) >= 10
    for n in names:
        assert hasattr(lib, n), n
    assert sorted(engine.EXPORTS) == names


def test_function_signatures_match_header():
    protos = _header_prototypes()
    assert sorted(protos) == _header_functions()
    for name, (ret, params) in protos.items():
        restype, argtypes = engine.ABI[name]
        assert _ctypes_kind(restype) == _c_kind(ret), (name, ret, restype)
        assert [_ctypes_kind(t) for t in argtypes] == [_c_kind(p) for p in params], (name, params, argtypes)


# ctypes mirror of every struct the Python side passes through the C-ABI
_MIRRORS = {"swb_params": engine.Params, "swb_result": engine.Result, "swb_solve_args": engine.SolveArgs,
            "swb_round_args": engine.RoundArgs, "swb_market_args": engine.MarketArgs,
            "swb_gavel_round_args": engine.GavelRoundArgs, "swb_sim_trace": engine.SimTrace,
            "swb_sim_dynamic": engine.SimDynamic, "swb_sim_scn": engine.SimScn}


def test_struct_layouts_match_header(tmp_path):
    assert engine.load_library().swb_version() >= 101
    cc = shutil.which("cc") or shutil.which("gcc")
    if cc is None:
        pytest.skip("no C compiler to read the header's struct layouts")
    lines = ["#include <stddef.h>", "#include <stdio.h>", '#include "swb200.h"', "int main(void) {"]
    for cname, mirror in _MIRRORS.items():
        lines.append(f'  printf("{cname} size %zu\\n", sizeof({cname}));')
        for field, _ in mirror._fields_:
            lines.append(f'  printf("{cname} {field} %zu\\n", offsetof({cname}, {field}));')
    lines += ["  return 0;", "}"]
    src, exe = tmp_path / "layouts.c", tmp_path / "layouts"
    src.write_text("\n".join(lines) + "\n")
    subprocess.check_call([cc, "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = {}
    for line in subprocess.check_output([str(exe)], text=True).splitlines():
        cname, key, value = line.split()
        got[(cname, key)] = int(value)
    for cname, mirror in _MIRRORS.items():
        assert C.sizeof(mirror) == got[(cname, "size")], cname
        for field, _ in mirror._fields_:
            assert getattr(mirror, field).offset == got[(cname, field)], (cname, field)


def test_no_gpu_fails_loudly():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(RuntimeError):
        engine.Engine(0)


def test_make_params():
    p = engine.make_params(32, 20, 120, 1e-3, 12.0, 1.0, [0.0, 0.2, 0.4, 0.6, 0.8, 1.0], {0.0: 1e-6}, 7)
    assert (p.ngpus, p.future_rounds, p.round_ptr, p.nbases) == (32, 20, 7, 6)
    assert abs(p.logv[0] - np.log(1e-6)) < 1e-15 and p.logv[5] == 0.0


class _FakeBackend(ShockwaveScheduler):
    """State machine only: the three backend hooks are replaced, nothing touches the GPU."""
    def _on_add(self, jobid, job): self.log.append(("add", jobid))
    def _on_remove(self, jobid): self.log.append(("rm", jobid))
    def _resolve(self, jobids, jobobjs):
        self.log.append(("solve", tuple(jobids), self.round_ptr, self.reestimate_share))
        return OrderedDict((self.round_ptr + t, list(jobids)) for t in range(self.future_nrounds))


class _J:
    def __init__(self): self.epoch_progress, self.waiting_delay, self.epochs = 0, 0, 10
    def set_epoch_progress(self, c): self.epoch_progress = c
    def reset_waiting_delay(self): self.waiting_delay = 0
    def add_waiting_delay(self, d): self.waiting_delay += d


def _mk():
    _FakeBackend.log = []
    return _FakeBackend(8, 16, OrderedDict(), 4, 120, ["GUROBI"], 1e-3, 24, 15, 30, [0.0, 1.0], {0.0: 1e-6}, 1e-3, 12.0, 1.0)


def test_resolve_and_cache_replay_state_machine():
    """shockwave.py:122-210: resolve set by add/remove/set_resolve, cleared by a solve; cached window
    replayed while round_ptr is inside it; reestimate_share only on add/remove."""
    sw = _mk()
    sw.add_metadata(1, _J()); sw.add_metadata(2, _J())
    assert sw.resolve and sw.reestimate_share
    assert sw.round_schedule() == [1, 2]
    assert not sw.resolve and not sw.reestimate_share
    n = len(sw.log)
    for _ in range(3):
        sw.increment_round_ptr()
        assert sw.round_schedule() == [1, 2]          # replay, no solve
    assert len(sw.log) == n
    sw.increment_round_ptr()                          # round 4 is outside the cached window [0,4)
    sw.round_schedule()
    assert sw.log[-1][0] == "solve" and sw.log[-1][3] is False
    sw.set_resolve(); sw.round_schedule()
    assert sw.log[-1][2] == 4 and sw.log[-1][3] is False
    sw.remove_metadata(1)
    assert sw.resolve and sw.reestimate_share and 1 in sw.completed_jobs
    assert sw.round_schedule() == [2] and sw.log[-1][3] is True
    with pytest.raises(AssertionError):
        sw.add_metadata(2, _J())
    sw.schedule_progress(2, 5); assert sw.metadata[2].epoch_progress == 5
    sw.deschedule_waiting_delay(2, 120); assert sw.metadata[2].waiting_delay == 120
    sw.deschedule_waiting_delay(99, 120)              # unknown id is ignored (shockwave.py:189-194)


def test_constructor_asserts_like_reference():
    with pytest.raises(AssertionError):
        _FakeBackend(0, 16, OrderedDict(), 4, 120, [], 1e-3, 24, 15, 30, [0.0, 1.0], {0.0: 1e-6}, 1e-3, 12.0, 1.0)
    with pytest.raises(AssertionError):
        _FakeBackend(8, 16, {}, 4, 120, [], 1e-3, 24, 15, 30, [0.0, 1.0], {0.0: 1e-6}, 1e-3, 12.0, 1.0)


def test_schedules_from_matrices_order():
    x = np.array([[1, 0], [0, 0], [0, 1], [0, 0]], dtype=np.uint8)
    bf = np.array([[0, 0], [1, 1], [0, 0], [1, 1]], dtype=np.uint8)
    s = schedules_from_matrices(x, bf, np.array([5.0, 9.0, 1.0, 9.0]), [10, 11, 12, 13], 7)
    assert s[7] == [10, 11, 13] and s[8] == [12, 11, 13]


@pytest.mark.parametrize("T", [1, 63, 64, 65, 127, 128])
def test_128_bit_mask_decoders(T):
    """engine.unpack_masks and the packed form of LazySchedules against the byte matrices, on both words of the mask"""
    from shockwave_b200.scheduler import LazySchedules
    rng = np.random.default_rng(T)
    J = 70
    x = (rng.random((J, T)) < 0.4).astype(np.uint8)
    bf = ((rng.random((J, T)) < 0.3) & (x == 0)).astype(np.uint8)

    def pack(m):
        full = np.zeros((J, 128), dtype=np.uint8)
        full[:, :T] = m
        w = (full.reshape(J, 2, 64).astype(np.uint64) << np.arange(64, dtype=np.uint64)).sum(axis=2, dtype=np.uint64)
        return np.ascontiguousarray(w)

    xm, bm = pack(x), pack(bf)
    assert np.array_equal(engine.unpack_masks(xm, T), x) and np.array_equal(engine.unpack_masks(bm, T), bf)
    assert np.array_equal(engine.unpack_masks(xm[None], T), x[None])
    if T > 64:
        assert xm[:, 1].any()
    bfkey = np.round(rng.uniform(0, 50, J))               # ties: the back-fill order must stay stable
    jobids = list(rng.permutation(1000)[:J])
    want = schedules_from_matrices(x, bf, bfkey, jobids, 17)
    got = LazySchedules(None, None, bfkey, jobids, 17, xmask=xm, bfmask=bm, T=T)
    assert list(got.keys()) == list(want.keys()) == list(range(17, 17 + T))
    for r in range(17, 17 + T):
        assert got[r] == want[r], r
