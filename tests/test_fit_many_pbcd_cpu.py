"""fit_many with solver="pbcd" (sparsepoly_b200/multi.py): validation and the memory bound come before any device
work or random draw, so these run without a GPU; plus the ctypes mirror of struct sp_pbcd_model."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest
import torch

import sparsepoly_b200 as S
from sparsepoly_b200 import _lib, multi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
X = np.random.RandomState(0).randn(20, 4)
Y = np.random.RandomState(1).randn(20)


def _fm(**kw):
    kw.setdefault("n_components", 3)
    kw.setdefault("solver", "pbcd")
    kw.setdefault("regularizer", "l21")
    return S.SparseFactorizationMachineRegressor(**kw)


@pytest.mark.parametrize("ests, match", [
    ([_fm(), _fm(solver="pcd", regularizer="l1")], "first estimator has solver='pbcd' supports solver='pbcd' only"),
    ([_fm(solver="pcd", regularizer="l1"), _fm()], "supports solver='pcd' only"),
    ([_fm(solver="psgd")], "supports solver='pcd' or solver='pbcd'"),
    ([_fm(solver="pcd", regularizer="l21")], "cannot be used with solver pcd"),
    ([_fm(regularizer="squaredl12")], "cannot be used with solver pbcd"),
    ([_fm(degree=3, regularizer="squaredl21")], "SquaredL21 supports only degree=2"),
    ([_fm(n_components=129)], "n_components=129 > 128"),
    ([_fm(degree=6)], "pbcd degree 6 is not supported"),
    ([S.SparseAllSubsetsRegressor(solver="pbcd", regularizer="omegati")], "cannot be used with solver pbcd"),
    ([_fm(), _fm(degree=3)], "degree must be equal"),
    ([_fm(shuffle=True)], "shares its random generator"),
])
def test_validation_errors_come_before_device_work(ests, match):
    with pytest.raises(ValueError, match=match):
        S.fit_many(ests, X, Y)
    for e in ests:                                      # nothing was drawn or fitted
        assert not hasattr(e, "P_")


def test_shared_generator_with_shuffle_is_refused():
    rs = np.random.RandomState(0)
    state = rs.get_state()[1].copy()
    with pytest.raises(ValueError, match="estimator 1 has shuffle=True"):
        S.fit_many([_fm(random_state=rs), _fm(shuffle=True, random_state=rs)], X, Y)
    assert np.array_equal(rs.get_state()[1], state)     # nothing drawn


def test_memory_bound_names_how_many_models_fit(monkeypatch):
    n, d, k = 1000, 50, 8
    Xb = np.random.RandomState(2).randn(n, d)
    yb = np.random.RandomState(3).randn(n)
    ests = [_fm(degree=3, n_components=k, regularizer="omegacs") for _ in range(10)]
    shared, model, plan = multi._pbcd_bytes(ests, n, d, n * d, True)
    assert model >= 8 * n * 2 * k                       # at least the A cache: n*(degree-1)*k doubles
    monkeypatch.setattr(multi, "_free_device_bytes", lambda: shared + 3 * model + model // 2)
    with pytest.raises(ValueError, match=r"10 pbcd models need .* 3 models of this shape fit"):
        S.fit_many(ests, Xb, yb)
    for e in ests:
        assert not hasattr(e, "P_")


def test_valid_call_needs_a_gpu():
    if torch.cuda.is_available():
        pytest.skip("needs a box without CUDA")
    ests = [_fm(shuffle=True, random_state=1), _fm(regularizer="omegacs", random_state=2), _fm(regularizer="l1")]
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        S.fit_many(ests, X, [Y, Y, Y])
    assert not any(hasattr(e, "P_") for e in ests)


def test_sp_pbcd_model_matches_the_header_layout(tmp_path):
    """sizeof / offsetof of struct sp_pbcd_model (compiled with gcc) against _lib.SpPbcdModel."""
    if shutil.which("gcc") is None:
        pytest.skip("gcc not available")
    cls = _lib.SpPbcdModel
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "sparsepoly_b200.h"', "int main(void) {",
             '  printf("size %zu\\n", sizeof(struct sp_pbcd_model));']
    for fname, _ in cls._fields_:
        lines.append(f'  printf("{fname} %zu\\n", offsetof(struct sp_pbcd_model, {fname}));')
    lines += ["  return 0;", "}"]
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)])
    got = dict((ln.split()[0], int(ln.split()[1])) for ln in subprocess.check_output([str(exe)], text=True).splitlines())
    assert got.pop("size") == C.sizeof(cls)
    assert got == {fname: getattr(cls, fname).offset for fname, _ in cls._fields_}
    assert _lib.SIGNATURES["sp_pbcd_epoch_multi"][1][3] == C.POINTER(cls)
