"""fit_many validation (sparsepoly_b200/multi.py): every error is raised before any device work, so these run
without a GPU; on a box without one, a valid call gets as far as the "no CPU fallback" error."""
import numpy as np
import pytest
import torch

import sparsepoly_b200 as S

X = np.random.RandomState(0).randn(20, 4)
Y = np.random.RandomState(1).randn(20)
YC = np.where(Y > 0, 1.0, -1.0)


def _fm(**kw):
    kw.setdefault("n_components", 3)
    return S.SparseFactorizationMachineRegressor(**kw)


@pytest.mark.parametrize("ests, y, match", [
    ([_fm(), _fm(solver="pbcd", regularizer="l1")], Y, "supports solver='pcd' only"),
    ([_fm(), S.SparseFactorizationMachineClassifier(n_components=3)], Y, "must be of one class"),
    ([_fm(), _fm(n_components=4)], Y, "n_components must be equal"),
    ([_fm(), _fm(degree=3, regularizer="l1")], Y, "degree must be equal"),
    ([_fm(), _fm(fit_linear=False)], Y, "fit_linear must be equal"),
    ([_fm(), _fm(fit_lower="augment")], Y, "fit_lower must be equal"),
    ([S.SparseFactorizationMachineClassifier(), S.SparseFactorizationMachineClassifier(loss="logistic")], YC,
     "loss must be equal"),
    ([_fm(), _fm()], [Y, Y, Y], "3 target arrays for 2 estimators"),
    ([_fm(), _fm(regularizer="l21")], Y, "cannot be used with solver pcd"),
    ([_fm(degree=3, regularizer="squaredl12")], Y, "SquaredL12 supports only degree=2"),
    ([_fm(degree=6, regularizer="l1")], Y, "degree 6 is not supported"),
    ([S.SparseAllSubsetsRegressor(regularizer="omegacs")], Y, "cannot be used with solver pcd"),
    ([_fm(shuffle=True)], Y, "shares its random generator"),
    ([_fm(shuffle=True, random_state=np.random.RandomState(0)), _fm(random_state=None)], Y, None),
    ([_fm(regularizer="foo")], Y, "Regularizer foo not supported"),
    ([_fm(init_lambdas="zeros")], Y, "Lambdas must be initialized"),
    ([object()], Y, "is not a SparseFactorizationMachine"),
])
def test_validation_errors_come_before_device_work(ests, y, match):
    if match is None:                                   # valid: shares nothing with a shuffling model
        if torch.cuda.is_available():
            pytest.skip("GPU present: the call would run")
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            S.fit_many(ests, X, y)
        return
    with pytest.raises(ValueError, match=match):
        S.fit_many(ests, X, y)
    for e in ests:                                      # nothing was drawn or fitted
        assert not hasattr(e, "P_")


def test_shared_generator_with_shuffle_is_refused():
    rs = np.random.RandomState(0)
    with pytest.raises(ValueError, match="estimator 1 has shuffle=True"):
        S.fit_many([_fm(random_state=rs), _fm(shuffle=True, random_state=rs)], X, Y)
    with pytest.raises(ValueError, match="shares its random generator"):
        S.fit_many([_fm(shuffle=True, random_state=np.random.mtrand._rand)], X, Y)


def test_classifier_targets_are_checked_per_model():
    est = S.SparseFactorizationMachineClassifier(n_components=2)
    with pytest.raises(TypeError, match="Only binary targets supported"):
        S.fit_many([est, S.SparseFactorizationMachineClassifier(n_components=2)], X, [YC, np.arange(20) % 3])


def test_empty_list():
    assert S.fit_many([], X, Y) == []


def test_valid_call_needs_a_gpu():
    if torch.cuda.is_available():
        pytest.skip("needs a box without CUDA")
    ests = [_fm(shuffle=True, random_state=1), _fm(regularizer="l1", random_state=2),
            S.SparseFactorizationMachineRegressor(n_components=3, regularizer="omegati")]
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        S.fit_many(ests, X, [Y, Y, Y])
    ovr = [S.SparseFactorizationMachineClassifier(n_components=2) for _ in range(3)]
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        S.fit_many(ovr, X, [YC, -YC, YC])
    assert all(hasattr(e, "label_binarizer_") for e in ovr)
