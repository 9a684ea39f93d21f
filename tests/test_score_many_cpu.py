"""decision_function_many / predict_many / score_many / objective_many (sparsepoly_b200/multi.py): every input check
comes before any device work, so these run without a GPU; plus the ctypes mirrors of the new header structs."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest
import torch
from sklearn.exceptions import NotFittedError

import sparsepoly_b200 as S
from sparsepoly_b200 import _lib, multi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
X = np.random.RandomState(0).randn(20, 4)
Y = np.random.RandomState(1).randn(20)
CALLS = [lambda e, X: S.decision_function_many(e, X), lambda e, X: S.predict_many(e, X),
         lambda e, X: S.score_many(e, X, Y), lambda e, X: S.objective_many(e, X, Y)]
NAMES = ["decision_function_many", "predict_many", "score_many", "objective_many"]


def _fitted(cls=S.SparseFactorizationMachineRegressor, d=4, **kw):
    e = cls(**kw)
    k = e.n_components
    if hasattr(e, "degree"):
        e.P_ = np.zeros((e.degree - 1 if e.fit_lower == "explicit" else 1, k, d))
        e.w_ = np.zeros(d)
    else:
        e.P_ = np.zeros((k, d))
    e.lams_ = np.ones(k)
    return e


def _no_device(monkeypatch):
    def refuse(*a, **k):
        raise AssertionError("device work before the checks")
    monkeypatch.setattr(multi, "_free_device_bytes", refuse)
    monkeypatch.setattr(multi, "DeviceDataset", refuse)


@pytest.mark.parametrize("call, name", list(zip(CALLS, NAMES)), ids=NAMES)
@pytest.mark.parametrize("ests, err, match", [
    ([_fitted(), S.SparseFactorizationMachineRegressor()], NotFittedError, "estimator 1 is not fitted"),
    ([_fitted(), _fitted(S.SparseFactorizationMachineClassifier)], ValueError, "all estimators must be of one class"),
    ([_fitted(), _fitted(S.SparseAllSubsetsRegressor)], ValueError, "all estimators must be of one class"),
    ([_fitted(), _fitted(degree=3)], ValueError, "degree must be equal"),
    ([_fitted(), _fitted(n_components=3)], ValueError, "n_components must be equal"),
    ([_fitted(degree=3), _fitted(degree=3, fit_lower=None)], ValueError, "fit_lower must be equal"),
    ([_fitted(), _fitted(fit_linear=False)], ValueError, "fit_linear must be equal"),
    ([_fitted(S.SparseAllSubsetsRegressor), _fitted(S.SparseAllSubsetsRegressor, n_components=5)], ValueError,
     "n_components must be equal"),
    ([_fitted(d=5)], ValueError, "X has 4 features; estimator 0 was fitted with 5"),
    ([_fitted(degree=4, fit_lower="augment", d=5)], ValueError, "X has 6 features after augmentation"),
    ([_fitted(), _fitted(n_components=2, d=4)], None, None),
    (["not an estimator"], ValueError, "str is not a SparseFactorizationMachine"),
])
def test_validation_errors_come_before_device_work(monkeypatch, call, name, ests, err, match):
    _no_device(monkeypatch)
    if err is None:                                     # a valid call reaches the device
        with pytest.raises(AssertionError, match="device work"):
            call(ests, X)
        return
    with pytest.raises(err, match=f"{name}: {match}" if not match.startswith("all") else match):
        call(ests, X)


def test_mismatched_model_arrays_are_refused(monkeypatch):
    _no_device(monkeypatch)
    e = _fitted()
    e.lams_ = np.ones(3)
    with pytest.raises(ValueError, match="estimator 1 has P_"):
        S.decision_function_many([_fitted(), e], X)
    e = _fitted(degree=3)
    e.P_ = e.P_[:1]
    with pytest.raises(ValueError, match="estimator 0 has P_"):
        S.predict_many([e], X)


@pytest.mark.parametrize("call", [S.score_many, S.objective_many])
def test_targets_are_checked_before_device_work(monkeypatch, call):
    _no_device(monkeypatch)
    ests = [_fitted(), _fitted()]
    with pytest.raises(ValueError, match="3 target arrays for 2 estimators"):
        call(ests, X, [Y, Y, Y])
    with pytest.raises(ValueError, match="target 1 has 19 samples and X has 20"):
        call(ests, X, [Y, Y[:19]])
    with pytest.raises(ValueError, match="target 0 has 21 samples and X has 20"):
        call(ests, X, np.append(Y, 0.0))


def test_empty_estimator_list():
    assert S.decision_function_many([], X).shape == (0, 20)
    assert S.predict_many([], X).shape == (0, 20)
    assert S.score_many([], X, Y).shape == (0,)
    assert S.objective_many([], X, Y) == []


def test_valid_call_needs_a_gpu():
    if torch.cuda.is_available():
        pytest.skip("needs a box without CUDA")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        S.decision_function_many([_fitted(), _fitted()], X)


@pytest.mark.parametrize("struct, cls, fn, arg", [
    ("sp_predict_model", _lib.SpPredictModel, "sp_predict_multi", 1),
    ("sp_loss_entry", _lib.SpLossEntry, "sp_loss_sum_multi", 0),
    ("sp_sqnorm_entry", _lib.SpSqnormEntry, "sp_sqnorm_multi", 0),
    ("sp_reg_entry", _lib.SpRegEntry, "sp_reg_eval_multi", 0),
])
def test_new_structs_match_the_header_layout(tmp_path, struct, cls, fn, arg):
    """sizeof / offsetof of each new header struct (compiled with gcc) against its ctypes mirror, and the table
    capacities _lib assumes."""
    if shutil.which("gcc") is None:
        pytest.skip("gcc not available")
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "sparsepoly_b200.h"', "int main(void) {",
             f'  printf("size %zu\\n", sizeof(struct {struct}));',
             '  printf("predict_max %d\\n", SP_PREDICT_MAX_MODELS);',
             '  printf("objective_max %d\\n", SP_OBJECTIVE_MAX_ENTRIES);']
    for fname, _ in cls._fields_:
        lines.append(f'  printf("{fname} %zu\\n", offsetof(struct {struct}, {fname}));')
    lines += ["  return 0;", "}"]
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)])
    got = dict((ln.split()[0], int(ln.split()[1])) for ln in subprocess.check_output([str(exe)], text=True).splitlines())
    assert got.pop("size") == C.sizeof(cls)
    assert got.pop("predict_max") == _lib.PREDICT_MAX_MODELS
    assert got.pop("objective_max") == _lib.OBJECTIVE_MAX_ENTRIES
    assert got == {fname: getattr(cls, fname).offset for fname, _ in cls._fields_}
    assert _lib.SIGNATURES[fn][1][arg] == C.POINTER(cls)
