"""fit_many with solver="pbcd" (sparsepoly_b200/multi.py, sp_pbcd_epoch_multi in csrc/pbcd.cu) against separate
fits: every model of a call must be bit-identical to est.fit(X, y_i) alone with the cluster sweep and the same
geometry."""
import contextlib
import ctypes as C
import io
import warnings

import numpy as np
import pytest
import scipy.sparse as sp
from sklearn.base import clone

import sparsepoly_b200 as S
from sparsepoly_b200 import _lib, synth

pytestmark = pytest.mark.gpu

FM_R, FM_C = S.SparseFactorizationMachineRegressor, S.SparseFactorizationMachineClassifier
AS_R, AS_C = S.SparseAllSubsetsRegressor, S.SparseAllSubsetsClassifier


@pytest.fixture(autouse=True)
def _cluster_sweep(monkeypatch):
    monkeypatch.setenv("SPARSEPOLY_B200_SWEEP", "cluster")


def _data(n=80, d=14, dense=False, seed=0):
    rng = np.random.RandomState(seed)
    X = synth.uniform_sparse(n, d, 5, seed)
    if dense:
        X = X.toarray() + 0.1 * rng.randn(n, d)
    y = rng.randn(n)
    return X, y, np.where(y > 0, 1.0, -1.0)


def _run(fn):
    """(result, stdout, convergence warnings) of fn()."""
    out = io.StringIO()
    with warnings.catch_warnings(record=True) as w, contextlib.redirect_stdout(out):
        warnings.simplefilter("always")
        r = fn()
    return r, out.getvalue(), [str(x.message) for x in w if "converge" in str(x.message)]


def _single(est, X, y):
    e = clone(est)
    _run(lambda: e.fit(X, y))
    return e


def _assert_same(got, want):
    assert np.array_equal(got.P_, want.P_)
    if hasattr(want, "w_"):
        assert np.array_equal(got.w_, want.w_)
    assert np.array_equal(got.lams_, want.lams_)
    assert got.n_iter_ == want.n_iter_
    if hasattr(want, "label_binarizer_"):
        assert np.array_equal(got.label_binarizer_.classes_, want.label_binarizer_.classes_)


def _check_many(ests, X, ys):
    fitted, _, _ = _run(lambda: S.fit_many([clone(e) for e in ests], X, ys))
    for e, f, yi in zip(ests, fitted, ys):
        _assert_same(f, _single(e, X, yi))
    return fitted


@pytest.mark.parametrize("dense", [False, True])
def test_mixed_grid_fm_degree2(dense):
    X, y, yc = _data(dense=dense)
    for cls, loss, yy in ((FM_R, "squared", y), (FM_C, "logistic", yc), (FM_C, "squared_hinge", yc)):
        kw = {} if cls is FM_R else {"loss": loss}
        ests = [cls(degree=2, n_components=3, solver="pbcd", regularizer=reg, alpha=a, beta=b, gamma=g, eta0=eta,
                    mean=mean, init_lambdas=lam, max_iter=3, tol=-1, random_state=i, **kw)
                for i, (reg, a, b, g, eta, mean, lam) in enumerate([
                    ("l1", 0.1, 0.5, 0.01, 1.0, False, "ones"),
                    ("l21", 1.0, 0.1, 0.05, 0.5, False, "random_signs"),
                    ("squaredl21", 0.01, 1e-3, 1e-4, 1.0, True, "ones"),
                    ("omegacs", 0.1, 0.1, 1e-3, 0.7, False, "random_signs"),
                    ("l1", 1.0, 0.0, 0.0, 1.0, False, "random_signs")])]
        fitted = _check_many(ests, X, [yy] * len(ests))
        assert all(np.any(f.P_ != 0) for f in fitted[:4])


@pytest.mark.parametrize("degree,fit_lower,fit_linear", [(3, "explicit", True), (3, "augment", True),
                                                         (3, None, False), (4, "explicit", False),
                                                         (4, "augment", False), (5, "explicit", True),
                                                         (5, None, True)])
def test_mixed_grid_higher_degrees(degree, fit_lower, fit_linear):
    X, y, yc = _data(dense=degree == 4)
    ests = [FM_C(degree=degree, loss="logistic", n_components=3, solver="pbcd", regularizer=reg, fit_lower=fit_lower,
                 fit_linear=fit_linear, beta=b, gamma=g, max_iter=3, tol=-1, random_state=i,
                 init_lambdas="random_signs" if i % 2 else "ones")
            for i, (reg, b, g) in enumerate([("l1", 0.1, 0.01), ("omegacs", 0.5, 1e-3), ("l21", 0.1, 1e-2),
                                             ("l1", 1e-3, 0.0)])]
    _check_many(ests, X, [yc] * len(ests))


@pytest.mark.parametrize("cls", [AS_R, AS_C])
def test_mixed_grid_all_subsets(cls):
    X, y, yc = _data()
    yy = y if cls is AS_R else yc
    kw = {} if cls is AS_R else {"loss": "squared_hinge"}
    ests = [cls(n_components=4, solver="pbcd", regularizer=reg, beta=b, gamma=g, eta0=eta, mean=mean, max_iter=3,
                tol=-1, random_state=i, **kw)
            for i, (reg, b, g, eta, mean) in enumerate([("l1", 0.1, 0.01, 0.1, False), ("omegacs", 1.0, 1e-3, 0.5, False),
                                                        ("l21", 1e-3, 1e-5, 0.1, True), ("omegacs", 0.1, 1e-2, 0.1, True)])]
    _check_many(ests, X, [yy] * len(ests))


@pytest.mark.parametrize("k", [3, 33, 64, 128], ids=["KCH1", "KCH2-33", "KCH2-64", "KCH4"])
def test_component_blocks(k):
    X, y, _ = _data(n=60, d=10)
    ests = [FM_R(degree=2, n_components=k, solver="pbcd", regularizer=reg, beta=0.1, gamma=g, max_iter=2, tol=-1,
                 random_state=i, init_lambdas="random_signs")
            for i, (reg, g) in enumerate([("l21", 1e-2), ("squaredl21", 1e-3), ("omegacs", 1e-4), ("l1", 1e-3)])]
    _check_many(ests, X, [y] * len(ests))
    a = [AS_R(n_components=k, solver="pbcd", regularizer=reg, beta=0.1, gamma=1e-3, max_iter=2, tol=-1,
              random_state=i) for i, reg in enumerate(["omegacs", "l21"])]
    _check_many(a, X, [y] * 2)


@pytest.mark.parametrize("n_cta,threads", [(1, 32), (2, 64), (4, 128), (16, 256)])
def test_geometries(monkeypatch, n_cta, threads):
    monkeypatch.setenv("SPARSEPOLY_B200_NCTA", str(n_cta))
    monkeypatch.setenv("SPARSEPOLY_B200_THREADS", str(threads))
    X, y, yc = _data(n=300, d=12)
    ests = [FM_C(degree=3, loss="squared_hinge", n_components=3, solver="pbcd", regularizer=reg, beta=0.1, gamma=g,
                 max_iter=3, tol=-1, random_state=i, shuffle=i == 1)
            for i, (reg, g) in enumerate([("l1", 0.01), ("omegacs", 1e-3), ("l21", 0.01)])]
    _check_many(ests, X, [yc] * 3)
    a = [AS_C(n_components=5, solver="pbcd", regularizer=reg, beta=0.1, gamma=1e-3, max_iter=3, tol=-1,
              random_state=i, shuffle=i == 0) for i, reg in enumerate(["omegacs", "l1"])]
    _check_many(a, X, [yc] * 2)


def test_staggered_stopping_shuffle_warm_start():
    X, y, _ = _data(n=120, d=20)
    warm = [FM_R(degree=2, n_components=4, solver="pbcd", regularizer="l21", beta=0.1, gamma=0.01, max_iter=2,
                 random_state=5, warm_start=True) for _ in range(2)]
    for e in warm:                                      # two identical fitted models, continued below
        _run(lambda: e.fit(X, y))
        e.set_params(max_iter=4)
    ests = [FM_R(degree=2, n_components=4, solver="pbcd", regularizer="l21", beta=1.0, gamma=1e9, max_iter=5,
                 tol=1e-300, random_state=0),                                     # every row dies
            FM_R(degree=2, n_components=4, solver="pbcd", regularizer="squaredl21", max_iter=10, tol=1e6,
                 random_state=1),                                                 # converges at epoch 1
            FM_R(degree=2, n_components=4, solver="pbcd", regularizer="omegacs", beta=0.1, gamma=1e-3, max_iter=7,
                 tol=1e-2, shuffle=True, random_state=2),
            FM_R(degree=2, n_components=4, solver="pbcd", regularizer="l1", beta=0.1, gamma=0.01, max_iter=9, tol=-1,
                 shuffle=True, random_state=np.random.RandomState(3)),
            FM_R(degree=2, n_components=4, solver="pbcd", regularizer="squaredl21", beta=0.3, gamma=0.1, max_iter=6,
                 tol=-1, random_state=4)]
    want, n_warn = [], 0
    for e in ests + [warm[0]]:
        w = clone(e) if e is not warm[0] else e
        n_warn += len(_run(lambda: w.fit(X, y))[2])
        want.append(w)
    got, _, warns = _run(lambda: S.fit_many([clone(e) for e in ests] + [warm[1]], X, y))
    for g, w in zip(got, want):
        _assert_same(g, w)
    assert got[1].n_iter_ == 0 and len({g.n_iter_ for g in got}) >= 4
    assert np.all(got[0].P_ == 0)
    assert len(warns) == n_warn


def test_recovery_branches_in_one_call():
    """omegacs negative dcache (omegacs.py:90-96, with its negative-cache recompute :75-76) and the squaredl21
    drift guard (squaredl21.py:49-50) in one call; the oracle run of the same models shows they are entered."""
    from oracle import oracle as O
    X = synth.uniform_sparse(300, 40, 6, 1)
    y = X @ np.random.RandomState(1).randn(40)
    kws = [dict(regularizer="omegacs", beta=0.1, gamma=0.3), dict(regularizer="squaredl21", beta=0.1, gamma=0.03),
           dict(regularizer="l21", beta=0.1, gamma=0.03)]
    common = dict(degree=2, n_components=4, solver="pbcd", alpha=0.1, max_iter=8, tol=-1.0, random_state=0)
    ests = [FM_R(**common, **kw) for kw in kws]
    _check_many(ests, X, [y] * 3)
    counts = []
    for kw in kws[:2]:
        O.branch_counts(reset=True)
        O.fit_fm(X, y, **common, **kw)
        counts.append(O.branch_counts())
    assert counts[0][0] >= 1 and counts[0][1] >= 1, counts
    assert counts[1][2] >= 1, counts


def test_more_clusters_than_fit_at_once():
    X, y, _ = _data(n=20, d=4, dense=True)
    rng = np.random.RandomState(11)
    ests = [FM_R(degree=2, n_components=3, solver="pbcd",
                 regularizer=("l1", "l21", "squaredl21", "omegacs")[i % 4],
                 beta=float(rng.choice([1e-3, 0.1, 1.0])), gamma=float(rng.choice([0.0, 1e-3, 0.1])),
                 max_iter=int(rng.randint(1, 6)), tol=-1, random_state=i) for i in range(300)]
    fitted, _, _ = _run(lambda: S.fit_many([clone(e) for e in ests], X, y))
    for i in rng.choice(300, 20, replace=False):
        _assert_same(fitted[i], _single(ests[i], X, y))


def test_one_vs_rest_matches_onevsrest_classifier():
    from sklearn.multiclass import OneVsRestClassifier
    X, _, _ = _data(n=150, d=16)
    labels = np.random.RandomState(7).randint(0, 4, X.shape[0])
    est = FM_C(degree=2, n_components=3, solver="pbcd", regularizer="omegacs", beta=0.1, gamma=1e-3, max_iter=4,
               tol=-1, random_state=0, loss="logistic")
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        ovr = OneVsRestClassifier(est).fit(X, labels)
    Y = ovr.label_binarizer_.transform(labels)
    Y = Y.toarray() if sp.issparse(Y) else Y
    fitted, _, _ = _run(lambda: S.fit_many([clone(est) for _ in range(4)], X, [Y[:, c] for c in range(4)]))
    for c in range(4):
        assert np.array_equal(fitted[c].P_, ovr.estimators_[c].P_)
        assert np.array_equal(fitted[c].w_, ovr.estimators_[c].w_)
        assert np.array_equal(fitted[c].decision_function(X), ovr.estimators_[c].decision_function(X))


def test_against_the_oracle():
    from oracle import oracle as O
    X, y, yc = _data(n=100, d=15)
    kws = [dict(regularizer="omegacs", beta=0.1, gamma=1e-3), dict(regularizer="squaredl21", beta=0.5, gamma=0.05),
           dict(regularizer="l21", beta=0.2, gamma=0.02, shuffle=True), dict(regularizer="l1", beta=0.1, gamma=1e-2)]
    ests = [FM_C(degree=2, loss="logistic", n_components=3, solver="pbcd", max_iter=3, tol=-1, random_state=i, **kw)
            for i, kw in enumerate(kws)]
    fitted, _, _ = _run(lambda: S.fit_many(ests, X, yc))
    for i, (kw, f) in enumerate(zip(kws, fitted)):
        out = O.fit_fm(X, yc, degree=2, loss="logistic", n_components=3, solver="pbcd", max_iter=3, tol=-1,
                       random_state=i, **kw)
        err = np.max(np.abs(f.P_ - out["P_"])) / max(np.max(np.abs(out["P_"])), 1e-300)
        assert err <= 1e-9, (i, err)
        assert np.array_equal(f.P_ != 0, out["P_"] != 0)
        want = O.objective_fm(X, yc, out["P_"], out["w_"], f.lams_, degree=f.degree, loss=f.loss,
                              regularizer=f.regularizer, alpha=f.alpha, beta=f.beta, gamma=f.gamma, mean=f.mean,
                              fit_lower=f.fit_lower, fit_linear=f.fit_linear)
        got = S.objective(f, X, f.label_binarizer_.inverse_transform(yc > 0))
        for part in ("loss", "l2_w", "l2_P", "omega", "total"):
            assert abs(got[part] - want[part]) <= 1e-9 * max(abs(want[part]), 1e-300), (part, got, want)
    for i, reg in enumerate(["omegacs", "l21"]):
        a = S.fit_many([AS_R(n_components=3, solver="pbcd", regularizer=reg, beta=0.1, gamma=1e-3, max_iter=3,
                             tol=-1, random_state=4)], X, y)[0]
        out = O.fit_all_subsets(X, y, n_components=3, solver="pbcd", regularizer=reg, beta=0.1, gamma=1e-3,
                                max_iter=3, tol=-1, random_state=4)
        err = np.max(np.abs(a.P_ - out["P_"])) / max(np.max(np.abs(out["P_"])), 1e-300)
        assert err <= 1e-9 and np.array_equal(a.P_ != 0, out["P_"] != 0), (reg, err)


def _launches(ests, X, y):
    lib = _lib.load()
    lib.sp_profile_enable(1)
    try:
        _run(lambda: S.fit_many(ests, X, y))
        ms, n = (C.c_double * 8)(), (C.c_longlong * 8)()
        _lib.check(lib.sp_profile_collect(ms, n))
    finally:
        lib.sp_profile_enable(0)
    return np.array(n[:])


@pytest.mark.parametrize("n_models", [1, 50])
def test_launches_are_shared(n_models):
    X, y, _ = _data(n=100, d=10, dense=True)
    k = 4

    def ests(epochs):
        return [FM_R(degree=3, n_components=k, solver="pbcd", regularizer=("omegacs", "l1", "l21")[i % 3],
                     beta=0.1 * (i + 1), gamma=1e-3, max_iter=epochs, tol=-1, random_state=i) for i in range(n_models)]
    # per epoch = the difference of two runs (the set-up predictions are per model, not per epoch)
    per_epoch = (_launches(ests(4), X, y) - _launches(ests(2), X, y)) / 2
    assert per_epoch[3] == 2                       # pbcd sweeps: one per block order (explicit degree 2, then 3)
    assert per_epoch[2] == 1                       # the linear sub-epoch
    assert per_epoch[0] == 2                       # rows: one cache precompute per order
    assert per_epoch[1] == 4                       # regcache: row norms + regularizer caches, per order


def test_callbacks_and_verbose_per_model():
    X, y, _ = _data()
    seen = {}

    def make_cb(name, stop_at):
        def cb(est):
            seen.setdefault(name, []).append((est.P_.copy(), est.w_.copy()))
            return True if len(seen[name]) == stop_at else None
        return cb

    def ests(tag):
        return [FM_R(n_components=3, solver="pbcd", regularizer="l21", beta=0.1, gamma=0.01, max_iter=6, tol=-1,
                     random_state=0, callback=make_cb(tag + "a", 3), n_calls=1, verbose=True),
                FM_R(n_components=3, solver="pbcd", regularizer="omegacs", beta=0.1, gamma=1e-3, max_iter=5, tol=-1,
                     random_state=1, verbose=True),
                FM_R(n_components=3, solver="pbcd", regularizer="squaredl21", max_iter=8, tol=-1, random_state=2,
                     callback=make_cb(tag + "c", 100), n_calls=2)]
    single = ests("s")
    outs, warns = "", []
    for e in single:
        _, o, w = _run(lambda: e.fit(X, y))
        outs, warns = outs + o, warns + w
    got, out_many, warns_many = _run(lambda: S.fit_many(ests("m"), X, y))
    for g, s in zip(got, single):
        _assert_same(g, s)
    assert got[0].n_iter_ == 2 and got[1].n_iter_ == 4
    assert out_many == outs and warns_many == warns
    for name in ("a", "c"):
        assert len(seen["m" + name]) == len(seen["s" + name])
        for (pm, wm), (ps, ws) in zip(seen["m" + name], seen["s" + name]):
            assert np.array_equal(pm, ps) and np.array_equal(wm, ws)


def test_errors_then_recovery():
    X, y, _ = _data()
    with pytest.raises(ValueError, match="supports solver='pbcd' only"):
        S.fit_many([FM_R(solver="pbcd", regularizer="l1"), FM_R()], X, y)
    with pytest.raises(ValueError, match="n_components=129"):
        S.fit_many([FM_R(solver="pbcd", regularizer="l1", n_components=129)], X, y)
    _check_many([FM_R(n_components=2, solver="pbcd", regularizer="l21", max_iter=2, random_state=0),
                 FM_R(n_components=2, solver="pbcd", regularizer="omegacs", max_iter=3, random_state=1)], X, [y, y])
