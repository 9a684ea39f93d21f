"""decision_function_many / predict_many / score_many / objective_many (sparsepoly_b200/multi.py, sp_predict_multi and
the *_multi reductions of csrc/objective.cu) against the single-model calls: every row, score and objective part must
be bit-identical to the estimator's own decision_function / predict / score and to objective(est, X, y)."""
import ctypes as C

import numpy as np
import pytest
import scipy.sparse as sp
from sklearn.base import clone

import sparsepoly_b200 as S
from sparsepoly_b200 import _lib, multi, synth

pytestmark = pytest.mark.gpu

FM_R, FM_C = S.SparseFactorizationMachineRegressor, S.SparseFactorizationMachineClassifier
AS_R, AS_C = S.SparseAllSubsetsRegressor, S.SparseAllSubsetsClassifier
REGS = ("l1", "l21", "squaredl12", "squaredl21", "omegati", "omegacs")


@pytest.fixture(autouse=True)
def _quiet(recwarn):
    yield                                             # convergence warnings of the short fits are expected


def _data(n=80, d=14, dense=False, seed=0):
    rng = np.random.RandomState(seed)
    X = synth.uniform_sparse(n, d, 5, seed)
    if dense:
        X = X.toarray() + 0.1 * rng.randn(n, d)
    y = rng.randn(n)
    return X, y


def _hand(cls, d, seed, **kw):
    """A model whose P_ / w_ / lams_ are set by hand (lams_ of mixed sign)."""
    rng = np.random.RandomState(seed)
    e = cls(**kw)
    k = e.n_components
    if hasattr(e, "degree"):
        n_orders = e.degree - 1 if e.fit_lower == "explicit" else 1
        e.P_ = 0.3 * rng.randn(n_orders, k, d)
        e.w_ = 0.1 * rng.randn(d)
    else:
        e.P_ = 0.3 * rng.randn(k, d)
    e.lams_ = np.where(rng.rand(k) < 0.5, -1.0, 1.0)
    return e


def _width(e, X):
    d = X.shape[1]
    return d + multi._n_dummies(e) if hasattr(e, "degree") else d


def _check(ests, X, ys, scores=True):
    """Every *_many call on (X, ys) against the single-model calls, exactly."""
    ys_list = ys if isinstance(ys, list) else [ys] * len(ests)
    dec = S.decision_function_many(ests, X)
    assert dec.shape == (len(ests), X.shape[0])
    pred = S.predict_many(ests, X)
    objs = S.objective_many(ests, X, ys)
    for b, e in enumerate(ests):
        assert np.array_equal(dec[b], e._predict(X)), b
        assert np.array_equal(pred[b], e.predict(X)), b
        assert objs[b] == S.objective(e, X, ys_list[b]), b
    if scores:
        sc = S.score_many(ests, X, ys)
        assert sc.shape == (len(ests),)
        for b, e in enumerate(ests):
            assert sc[b] == e.score(X, ys_list[b]), b
    return dec


def test_fit_many_grid_dense_csr_csc():
    rng = np.random.RandomState(0)
    X = rng.randn(260, 100) * (rng.rand(260, 100) < 0.3)
    y = rng.randn(260)
    Xtr, ytr, Xte, yte = X[:200], y[:200], X[200:], y[200:]
    ests = [FM_R(degree=2, n_components=30, regularizer=reg, beta=beta, gamma=gamma, max_iter=3, tol=-1,
                 random_state=0)
            for reg in ("l1", "squaredl12", "omegati") for gamma in (1e-3, 1e-2, 0.1, 1.0) for beta in (0.1, 1.0)]
    S.fit_many(ests, Xtr, ytr)
    assert len(ests) == 24
    for Xh in (Xte, sp.csr_matrix(Xte), sp.csc_matrix(Xte)):
        _check(ests, Xh, yte)


FM_VARIANTS = [dict(degree=m, n_components=5) for m in (2, 3, 4, 5)] + \
    [dict(degree=3, n_components=5, fit_lower=fl) for fl in ("augment", None)] + \
    [dict(degree=3, n_components=5, fit_lower="augment", fit_linear=False),
     dict(degree=3, n_components=5, fit_linear=False), dict(degree=2, n_components=5, fit_linear=False)] + \
    [dict(degree=2, n_components=k) for k in (16, 30, 64, 100)] + [dict(degree=3, n_components=64)]


@pytest.mark.parametrize("kw", FM_VARIANTS, ids=lambda kw: "-".join(f"{a}{b}" for a, b in kw.items()))
def test_fm_instantiations(kw):
    X, y = _data(n=90, d=14)
    Xte, yte = _data(n=70, d=14, seed=5)
    fitted = FM_R(regularizer="omegati", beta=0.1, gamma=0.01, max_iter=2, tol=-1, random_state=1, **kw).fit(X, y)
    d = _width(fitted, X)
    ests = [fitted] + [_hand(FM_R, d, s, regularizer=REGS[s % 6], mean=bool(s % 2), alpha=0.5, beta=0.2, gamma=0.3,
                             **kw) for s in range(5)]
    _check(ests, Xte, yte)


@pytest.mark.parametrize("cls", [AS_R, AS_C])
def test_all_subsets(cls):
    X, y = _data(n=90, d=12)
    Xte, yte = _data(n=60, d=12, seed=3)
    if cls is AS_C:
        y, yte = np.where(y > 0, 1, -1), np.where(yte > 0, 1, -1)
    ests = [cls(n_components=k, solver=solver, regularizer=reg, beta=0.1, gamma=0.01, max_iter=2, tol=-1, mean=mean,
                random_state=0).fit(0.5 * X, y)
            for k in (6,) for solver, reg, mean in (("pcd", "omegati", False), ("pbcd", "omegacs", True),
                                                    ("pcd", "omegati", True))]
    if cls is AS_R:
        ests += [_hand(AS_R, 12, s, n_components=6, regularizer=("omegati", "omegacs")[s % 2]) for s in range(3)]
        ests[-1].P_ *= 0.1
    _check(ests, 0.5 * Xte, yte)


def test_models_from_every_source():
    X, y = _data(n=120, d=16)
    Xte, yte = _data(n=50, d=16, seed=7)
    base = dict(degree=2, n_components=4, beta=0.1, gamma=0.01, max_iter=3, tol=-1, random_state=0)
    ests = [FM_R(solver="pcd", regularizer="l1", **base).fit(X, y),
            FM_R(solver="pcd", regularizer="squaredl12", mean=True, **base).fit(X, y),
            FM_R(solver="pbcd", regularizer="l21", **base).fit(X, y),
            FM_R(solver="pbcd", regularizer="squaredl21", mean=True, **base).fit(X, y),
            FM_R(solver="pbcd", regularizer="omegacs", **base).fit(X, y),
            FM_R(solver="psgd", regularizer="squaredl12", batch_size=16, **base).fit(X, y),
            FM_R(solver="psgd", regularizer="l21", batch_size=16, **base).fit(X, y)]
    stream = FM_R(solver="psgd", regularizer="l1", batch_size=16, **base)
    for i in range(0, 120, 40):
        stream.partial_fit(X[i:i + 40], y[i:i + 40])
    warm = FM_R(solver="pcd", regularizer="omegati", warm_start=True, **base).fit(X, y)
    warm.set_params(gamma=0.1).fit(X, y)
    many = [clone(FM_R(solver="pcd", regularizer="omegati", **base)) for _ in range(2)]
    S.fit_many(many, X, [y, -y])
    hand = _hand(FM_R, 16, 3, degree=2, n_components=4, regularizer="omegati", mean=True)
    ests += [stream, warm] + many + [hand]
    _check(ests, Xte, yte)
    _check(ests, Xte, [yte * (b + 1) for b in range(len(ests))])


def test_classifiers_with_different_labels_and_one_vs_rest():
    X, y = _data(n=120, d=14)
    Xte, yte = _data(n=60, d=14, seed=9)
    pos = y > 0
    labels = [(0, 1), (-1, 1), (3, 7), ("a", "b")]
    ests, ys = [], []
    for lo, hi in labels:
        lab = np.where(pos, hi, lo)
        ests.append(FM_C(n_components=4, regularizer="squaredl12", beta=0.1, gamma=0.01, max_iter=3, tol=-1,
                         loss=("squared_hinge", "logistic", "squared", "squared_hinge")[len(ests)],
                         random_state=0).fit(X, lab))
        ys.append(np.where(yte > 0, hi, lo))
    pred = S.predict_many(ests, Xte)
    for b, e in enumerate(ests):
        assert np.array_equal(pred[b], e.predict(Xte))
    _check(ests, Xte, ys)
    # one-vs-rest: 4 classes, one binary model per class, class = argmax of the decision functions
    cls = np.digitize(y, [-1.0, 0.0, 1.0])
    cls_te = np.digitize(yte, [-1.0, 0.0, 1.0])
    ovr = [FM_C(n_components=4, regularizer="omegati", beta=0.1, gamma=0.01, max_iter=3, tol=-1, random_state=c)
           for c in range(4)]
    S.fit_many(ovr, X, [np.where(cls == c, 1, -1) for c in range(4)])
    targets = [np.where(cls_te == c, 1, -1) for c in range(4)]
    dec = _check(ovr, Xte, targets)
    single = np.stack([e.decision_function(Xte) for e in ovr])
    assert np.array_equal(dec.argmax(axis=0), single.argmax(axis=0))


def test_chunking_does_not_change_results(monkeypatch):
    X, y = _data(n=70, d=14)
    ests = [_hand(FM_R, 14, s, degree=3, n_components=8, regularizer=REGS[s % 6], mean=bool(s % 2)) for s in range(8)]
    whole = (S.decision_function_many(ests, X), S.predict_many(ests, X), S.score_many(ests, X, y),
             S.objective_many(ests, X, y))
    monkeypatch.setattr(multi, "SCORE_MAX_MODELS", 3)
    chunked = (S.decision_function_many(ests, X), S.predict_many(ests, X), S.score_many(ests, X, y),
               S.objective_many(ests, X, y))
    monkeypatch.setattr(multi, "SCORE_MAX_MODELS", 256)
    shared, model = multi._score_bytes(70, X.nnz, (2, 8, 14), True)
    monkeypatch.setattr(multi, "_free_device_bytes", lambda: shared + 3 * model + model // 2)
    by_memory = (S.decision_function_many(ests, X), S.predict_many(ests, X), S.score_many(ests, X, y),
                 S.objective_many(ests, X, y))
    for got in (chunked, by_memory):
        for a, b in zip(got[:3], whole[:3]):
            assert np.array_equal(a, b)
        assert got[3] == whole[3]
    monkeypatch.setattr(multi, "_free_device_bytes", lambda: shared + model // 2)
    with pytest.raises(ValueError, match="one model of this shape needs"):
        S.objective_many(ests, X, y)


def test_edge_cases():
    X, y = _data(n=40, d=10)
    ests = [_hand(FM_R, 10, s, degree=3, n_components=5, regularizer=REGS[s]) for s in range(4)]
    zero = _hand(FM_R, 10, 9, degree=3, n_components=5, regularizer="omegacs")
    zero.P_[...] = 0.0
    ests.append(zero)
    # 0 rows
    X0 = np.zeros((0, 10))
    assert S.decision_function_many(ests, X0).shape == (5, 0)
    assert S.predict_many(ests, X0).shape == (5, 0)
    objs0 = S.objective_many(ests, X0, np.zeros(0))
    full = S.objective_many(ests, X, y)
    for o0, o in zip(objs0, full):
        assert o0["loss"] == 0.0 and o0["l2_P"] == o["l2_P"] and o0["omega"] == o["omega"]
    # empty rows
    Xe = sp.csr_matrix(X)
    Xe = sp.vstack([Xe[:5], sp.csr_matrix((3, 10)), Xe[5:], sp.csr_matrix((2, 10))]).tocsr()
    ye = np.concatenate([y[:5], np.zeros(3), y[5:], np.ones(2)])
    _check(ests, Xe, ye)
    # one estimator, the zero model on its own
    _check(ests[:1], X, y)
    _check([zero], X, y)


def _rows_launches(fn):
    lib = _lib.load()
    lib.sp_profile_enable(1)
    try:
        fn()
        ms, n = (C.c_double * 8)(), (C.c_longlong * 8)()
        _lib.check(lib.sp_profile_collect(ms, n))
    finally:
        lib.sp_profile_enable(0)
    return n[0]


def _kernel_launches(fn):
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return sum(1 for ev in prof.events() if ev.device_type == torch.autograd.DeviceType.CUDA
               and "memcpy" not in ev.name.lower() and "memset" not in ev.name.lower())


@pytest.mark.parametrize("kw", [dict(degree=3, fit_lower="explicit"), dict(degree=2), dict(degree=4)])
def test_launches_are_shared(kw):
    X, y = _data(n=60, d=12)
    n_orders = kw["degree"] - 1
    _kernel_launches(lambda: S.objective_many([_hand(FM_R, 12, 0, n_components=6, **kw)], X, y))   # profiler warm-up
    one_kind, mixed = [], []
    for B in (1, 8, 64):
        ests = [_hand(FM_R, 12, s, n_components=6, regularizer=REGS[s % 6], **kw) for s in range(B)]
        assert _rows_launches(lambda: S.decision_function_many(ests, X)) == len(ests[0]._output_orders())
        ti = [_hand(FM_R, 12, s, n_components=6, regularizer="omegati", **kw) for s in range(B)]
        one_kind.append(_kernel_launches(lambda: S.objective_many(ti, X, y)))
        if B > 1:
            mixed.append(_kernel_launches(lambda: S.objective_many(ests, X, y)))
    assert one_kind[0] == one_kind[1] == one_kind[2], one_kind
    # column-fold and row-norm regularizers together: one more partial launch per order, whatever B is
    assert mixed == [one_kind[0] + n_orders] * 2, (mixed, one_kind)
