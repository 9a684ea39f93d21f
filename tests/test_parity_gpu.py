"""Parity of the CUDA backend (through the C ABI) against
  (1) the golden outputs of the unmodified reference (tests/golden, every solver x regularizer
      x loss x degree combination the reference tests cover, plus sparse inputs, shuffle,
      explicit / augmented lower orders, warm start), and
  (2) the pinned C oracle on larger seeded sparse problems, for several cluster geometries.
Tolerance: 1e-9 relative on coefficients / predictions (north_star), identical support sets."""
import os
import warnings

import numpy as np
import pytest
import scipy.sparse as sp

from golden_util import case_names, large_case_names, load_case, load_large_case, rel_err, same_support

pytestmark = pytest.mark.gpu

TOL = 1e-9


def _estimator(rec):
    import sparsepoly_b200 as S
    if rec["model"] == "fm":
        cls = S.SparseFactorizationMachineClassifier if rec["clf"] else S.SparseFactorizationMachineRegressor
    else:
        cls = S.SparseAllSubsetsClassifier if rec["clf"] else S.SparseAllSubsetsRegressor
    return cls(**rec["kw"])


def _fit(est, X, y, P_init=None):
    if P_init is not None:
        est.warm_start = True
        est.P_ = P_init.copy()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        est.fit(X, y)
    return est


@pytest.mark.parametrize("name", case_names())
def test_matches_reference_golden(name):
    rec, X, arr = load_case(name)
    est = _fit(_estimator(rec), X, arr["y"], arr.get("P_init"))
    assert rel_err(est.P_, arr["P_"]) <= TOL
    assert same_support(est.P_, arr["P_"])
    if "w_" in arr:
        assert rel_err(est.w_, arr["w_"]) <= TOL
    assert est.n_iter_ == int(arr["n_iter_"])
    if "it_" in arr:
        assert est.it_ == int(arr["it_"])
    pred = est.decision_function(arr["Xte"]) if rec["clf"] else est.predict(arr["Xte"])
    assert rel_err(pred, arr["pred_te"]) <= TOL
    _check_objective(est, X, arr["y"], arr["P_"], arr.get("w_"))


def _check_objective(est, X, y_pm1, P_ref, w_ref, tol=TOL):
    """Objective of the CUDA fit (device evaluator, sparsepoly_b200.objective) against the oracle's
    evaluation of the REFERENCE's (or the oracle's) fitted parameters: 1e-9 relative (north_star)."""
    from sparsepoly_b200.objective import objective
    from oracle import oracle as O
    y_user = est.label_binarizer_.inverse_transform(y_pm1 > 0) if hasattr(est, "label_binarizer_") else y_pm1
    got = objective(est, X, y_user)
    if hasattr(est, "degree"):
        w = w_ref if w_ref is not None else np.zeros(P_ref.shape[2])
        want = O.objective_fm(X, y_pm1, P_ref, w, est.lams_, degree=est.degree, loss=est.loss,
                              regularizer=est.regularizer, alpha=est.alpha, beta=est.beta,
                              gamma=est.gamma, mean=est.mean, fit_lower=est.fit_lower,
                              fit_linear=est.fit_linear)
    else:
        want = O.objective_all_subsets(X, y_pm1, P_ref, est.lams_, loss=est.loss,
                                       regularizer=est.regularizer, beta=est.beta, gamma=est.gamma,
                                       mean=est.mean)
    for part in ("loss", "l2_w", "l2_P", "omega", "total"):
        assert abs(got[part] - want[part]) <= tol * max(abs(want[part]), 1e-300), (part, got, want)
    return got


@pytest.mark.parametrize("n_cta,threads", [(2, 32), (4, 64), (8, 32), (16, 32), (1, 256), (2, 128)])
@pytest.mark.parametrize("name", ["pcd_fm_d3_omegati_logistic", "pcd_fm_sql12_squared",
                                  "pcd_all_omegati_squared_hinge", "pbcd_fm_d3_omegacs_logistic",
                                  "pbcd_fm_sql21", "pbcd_all_l21", "pcd_fm_d3_shuffle"])
def test_cluster_geometries_match_golden(name, n_cta, threads, monkeypatch):
    monkeypatch.setenv("SPARSEPOLY_B200_NCTA", str(n_cta))
    monkeypatch.setenv("SPARSEPOLY_B200_THREADS", str(threads))
    rec, X, arr = load_case(name)
    est = _fit(_estimator(rec), X, arr["y"], arr.get("P_init"))
    assert rel_err(est.P_, arr["P_"]) <= TOL
    assert same_support(est.P_, arr["P_"])
    if "w_" in arr:
        assert rel_err(est.w_, arr["w_"]) <= TOL


# ------------------------------------------------------------- pipelined window sweep (pcd_window.cu)
WINDOW_GEOMS = [(None, 0), (None, 1), (2, 1), (1, 0), (3, 0)]


@pytest.mark.parametrize("window,horizon", WINDOW_GEOMS)
@pytest.mark.parametrize("name", [n for n in case_names() if n.startswith("pcd")])
def test_window_sweep_matches_golden(name, window, horizon, monkeypatch):
    monkeypatch.setenv("SPARSEPOLY_B200_SWEEP", "window")
    monkeypatch.setenv("SPARSEPOLY_B200_HORIZON", str(horizon))
    monkeypatch.setenv("SPARSEPOLY_B200_NEAR", "2" if horizon else "1")
    if window is not None:
        monkeypatch.setenv("SPARSEPOLY_B200_WINDOW", str(window))
    rec, X, arr = load_case(name)
    est = _fit(_estimator(rec), X, arr["y"], arr.get("P_init"))
    assert est._dev_state["plan"].mode == "window"
    assert rel_err(est.P_, arr["P_"]) <= TOL
    assert same_support(est.P_, arr["P_"])
    if "w_" in arr:
        assert rel_err(est.w_, arr["w_"]) <= TOL
    assert est.n_iter_ == int(arr["n_iter_"])


WINDOW_ORACLE = [
    ("fm3_omegati_logistic", "anova", 3, True,
     dict(degree=3, loss="logistic", n_components=4, solver="pcd", regularizer="omegati", beta=1e-6,
          gamma=2e-9, alpha=1e-4, max_iter=2, tol=-1.0, random_state=0, mean=True, fit_lower="explicit")),
    ("fm2_sql12_squared", "anova", 2, False,
     dict(degree=2, n_components=4, solver="pcd", regularizer="squaredl12", beta=1e-5, gamma=1e-6,
          alpha=1e-3, max_iter=2, tol=-1.0, random_state=0, mean=True)),
    ("fm4_l1_sqhinge_shuffle", "anova", 2, True,
     dict(degree=4, loss="squared_hinge", n_components=3, solver="pcd", regularizer="l1", beta=1e-4,
          gamma=1e-5, alpha=1e-4, max_iter=2, tol=-1.0, random_state=0, mean=True, shuffle=True)),
]


@pytest.mark.parametrize("window,horizon,near", [(None, 1, 1), (None, 0, 2), (64, 0, 0), (8, 1, 2), (32, 0, 4)])
@pytest.mark.parametrize("tag,kernel,degree,clf,kw", WINDOW_ORACLE, ids=[c[0] for c in WINDOW_ORACLE])
def test_window_sweep_sparse_matches_oracle(tag, kernel, degree, clf, kw, window, horizon, near, monkeypatch):
    """columns share ~0.4 samples pairwise: most nonzeros are cold (bulk CTAs), the rest go through
    the engine's shared-memory slots; `near` = how far back a dependency is resolved by the chain
    warp itself"""
    monkeypatch.setenv("SPARSEPOLY_B200_SWEEP", "window" if window else "auto")
    monkeypatch.setenv("SPARSEPOLY_B200_HORIZON", str(horizon))
    monkeypatch.setenv("SPARSEPOLY_B200_NEAR", str(near))
    if window is not None:
        monkeypatch.setenv("SPARSEPOLY_B200_WINDOW", str(window))
    X, y = _problem(n=100000, d=5000, r=10, seed=5, kernel=kernel, degree=degree, clf=clf)
    est, out, frac = _compare_fm(kw, X, y)
    plan = est._dev_state["plan"]
    assert plan.mode == "window", plan.wplan.stats
    assert 0.0 < plan.wplan.stats["hot_frac"] < 0.6
    assert 0.01 < frac < 0.99
    print(tag, plan.wplan.stats, "nonzero fraction of P_", frac)


SPEC_CASES = [
    # (tag, degree of the planted target, clf, estimator kwargs): regimes in which (almost) every coordinate
    # sits at zero after the first epoch -> the window engine speculates on zero updates
    ("sql12_1pct", 2, False, dict(degree=2, n_components=4, solver="pcd", regularizer="squaredl12", beta=1e-5,
                                  gamma=4e-6, alpha=1e-3, max_iter=4, tol=-1.0, random_state=0, mean=True)),
    ("sql12_5pct", 2, False, dict(degree=2, n_components=4, solver="pcd", regularizer="squaredl12", beta=1e-5,
                                  gamma=1e-6, alpha=1e-3, max_iter=3, tol=-1.0, random_state=0, mean=True)),
    ("omegati_1pct", 2, False, dict(degree=2, n_components=4, solver="pcd", regularizer="omegati", beta=1e-5,
                                    gamma=1e-5, alpha=1e-3, max_iter=4, tol=-1.0, random_state=0, mean=True)),
    ("l1_all_zero", 2, False, dict(degree=2, n_components=4, solver="pcd", regularizer="l1", beta=1e-5,
                                   gamma=1e-4, alpha=1e-3, max_iter=3, tol=-1.0, random_state=0, mean=True)),
    ("fm3_omegati_logistic", 3, True,
     dict(degree=3, loss="logistic", n_components=4, solver="pcd", regularizer="omegati", beta=1e-6, gamma=1e-7,
          alpha=1e-4, max_iter=3, tol=-1.0, random_state=0, mean=True, fit_lower="explicit", shuffle=True)),
]


def _wspec_read():
    import ctypes as C
    from sparsepoly_b200 import _lib
    out = (C.c_ulonglong * 2)()
    _lib.check(_lib.load().sp_wspec_read(out))
    return int(out[0]), int(out[1])


@pytest.mark.parametrize("window", [None, 32])
@pytest.mark.parametrize("tag,degree,clf,kw", SPEC_CASES, ids=[c[0] for c in SPEC_CASES])
def test_window_sweep_zero_update_speculation(tag, degree, clf, kw, window, monkeypatch):
    """Sparse regimes: the engine's workers skip the per-record waits and the chain warp validates
    (pcd_window.cu, ZERO-UPDATE SPECULATION).  Results must equal the oracle's to 1e-9 and those of the
    non-speculative sweep to rounding, with identical supports."""
    monkeypatch.setenv("SPARSEPOLY_B200_SWEEP", "window" if window else "auto")
    if window is not None:
        monkeypatch.setenv("SPARSEPOLY_B200_WINDOW", str(window))
    X, y = _problem(n=100000, d=5000, r=10, seed=5, kernel="anova", degree=degree, clf=clf)
    _wspec_read()
    est, out, frac = _compare_fm(kw, X, y)
    n_spec, n_rej = _wspec_read()
    assert est._dev_state["plan"].mode == "window"
    if frac == 0.0:
        # every component is entirely zero after the first epoch: sp_pcd_epoch skips those sweeps exactly (dead-component
        # shortcut, pcd.cu), so there is nothing left to speculate on
        assert n_spec == 0
    else:
        assert n_spec > 0, "speculation never engaged"
        assert n_rej < n_spec
    print(tag, "nonzero fraction", frac, "speculated positions", n_spec, "rejected", n_rej)
    monkeypatch.setenv("SPARSEPOLY_B200_SPEC", "0")
    est0, _, _ = _compare_fm(kw, X, y)
    assert _wspec_read() == (0, 0)
    # (and with the dead-component shortcut disabled the sweeps run and give the same model)
    # same arithmetic per nonzero; only the order in which a column's hot terms are summed differs (in a
    # speculative window the workers sum all of them, otherwise the chain warp adds the "late" ones)
    assert rel_err(est.P_, est0.P_) <= 1e-11 and rel_err(est.w_, est0.w_) <= 1e-11
    assert np.array_equal(est.P_ != 0, est0.P_ != 0)


@pytest.mark.parametrize("horizon", [0, 1])
def test_window_sweep_all_subsets_matches_oracle(horizon, monkeypatch):
    import sparsepoly_b200 as S
    from oracle import oracle as O
    monkeypatch.setenv("SPARSEPOLY_B200_SWEEP", "auto")
    monkeypatch.setenv("SPARSEPOLY_B200_HORIZON", str(horizon))
    X, y = _problem(n=100000, d=4000, r=8, seed=3, kernel="all", degree=2, clf=True)
    kw = dict(loss="squared_hinge", n_components=4, solver="pcd", regularizer="omegati", beta=1e-4,
              gamma=1e-5, mean=True, max_iter=2, tol=-1.0, random_state=0)
    est = _fit(S.SparseAllSubsetsClassifier(**kw), X, y)
    assert est._dev_state["plan"].mode == "window"
    out = O.fit_all_subsets(X, y, **kw)
    assert rel_err(est.P_, out["P_"]) <= TOL
    assert same_support(est.P_, out["P_"])


@pytest.mark.parametrize("window,horizon", [(None, 0), (None, 1), (2, 1), (1, 0), (3, 0)])
@pytest.mark.parametrize("name", [n for n in case_names() if n.startswith("pbcd")])
def test_pbcd_window_sweep_matches_golden(name, window, horizon, monkeypatch):
    monkeypatch.setenv("SPARSEPOLY_B200_SWEEP", "window")
    monkeypatch.setenv("SPARSEPOLY_B200_HORIZON", str(horizon))
    if window is not None:
        monkeypatch.setenv("SPARSEPOLY_B200_WINDOW", str(window))
    rec, X, arr = load_case(name)
    est = _fit(_estimator(rec), X, arr["y"], arr.get("P_init"))
    assert est._dev_state["plan"].mode == "window"
    assert rel_err(est.P_, arr["P_"]) <= TOL
    assert same_support(est.P_, arr["P_"])
    if "w_" in arr:
        assert rel_err(est.w_, arr["w_"]) <= TOL
    assert est.n_iter_ == int(arr["n_iter_"])


PBCD_WINDOW_ORACLE = [
    ("fm2_omegacs", dict(degree=2, n_components=8, solver="pbcd", regularizer="omegacs", beta=1e-5, gamma=1e-7,
                         alpha=1e-4, max_iter=2, tol=-1.0, random_state=0, mean=True), 2, False),
    ("fm3_l21_logistic_explicit", dict(degree=3, loss="logistic", n_components=5, solver="pbcd", regularizer="l21",
                                       beta=1e-6, gamma=1e-7, alpha=1e-4, max_iter=2, tol=-1.0, random_state=0,
                                       mean=True, fit_lower="explicit"), 3, True),
    ("fm2_sql21_shuffle", dict(degree=2, n_components=32, solver="pbcd", regularizer="squaredl21", beta=1e-5,
                               gamma=1e-8, alpha=1e-4, max_iter=2, tol=-1.0, random_state=0, mean=True,
                               shuffle=True), 2, False),
]


@pytest.mark.parametrize("window,horizon", [(None, 0), (16, 1)])
@pytest.mark.parametrize("tag,kw,degree,clf", PBCD_WINDOW_ORACLE, ids=[c[0] for c in PBCD_WINDOW_ORACLE])
def test_pbcd_window_sweep_sparse_matches_oracle(tag, kw, degree, clf, window, horizon, monkeypatch):
    monkeypatch.setenv("SPARSEPOLY_B200_SWEEP", "window" if window else "auto")
    monkeypatch.setenv("SPARSEPOLY_B200_HORIZON", str(horizon))
    if window is not None:
        monkeypatch.setenv("SPARSEPOLY_B200_WINDOW", str(window))
    X, y = _problem(n=100000, d=5000, r=10, seed=6, kernel="anova", degree=degree, clf=clf)
    est, out, frac = _compare_fm(kw, X, y)
    plan = est._dev_state["plan"]
    assert plan.mode == "window", plan.wplan.stats
    print(tag, plan.wplan.stats, "nonzero fraction of P_", frac)


# ----------------------------------------------------------------------------- vs the C oracle
def _problem(n, d, r, seed, kernel, degree, clf):
    from sparsepoly_b200 import synth
    from oracle import oracle as O
    X = synth.uniform_sparse(n, d, r, seed)
    Pt = synth.planted_P(d, 3, seed + 1, frac_features=0.3, scale=0.5)
    if kernel == "anova":
        s = O.poly_predict(X, Pt, np.ones(3), "anova", degree)
    else:
        s = O.poly_predict(X, 0.3 * Pt, np.ones(3), "all-subsets")
    return X, synth.targets_from_scores(s, seed + 2, clf)


def _compare_fm(kw, X, y, tol=TOL):
    import sparsepoly_b200 as S
    from oracle import oracle as O
    clf = kw.get("loss", "squared") != "squared"
    cls = S.SparseFactorizationMachineClassifier if clf else S.SparseFactorizationMachineRegressor
    ekw = dict(kw)
    if not clf:
        ekw.pop("loss", None)
    est = _fit(cls(**ekw), X, y)
    okw = dict(kw)
    okw.setdefault("loss", "squared")
    out = O.fit_fm(X, y, **okw)
    assert rel_err(est.P_, out["P_"]) <= tol
    assert same_support(est.P_, out["P_"])
    assert rel_err(est.w_, out["w_"]) <= tol
    _check_objective(est, X, y, out["P_"], out["w_"], tol)
    frac = float(np.mean(out["P_"] != 0))
    return est, out, frac


CASES_ORACLE = [
    # scaled versions of the BASELINE configs (C1 full size; C2-C5 shrunk so the oracle takes seconds)
    ("C1", dict(n=10000, d=1000, r=50, seed=0, kernel="anova", degree=2, clf=False),
     dict(degree=2, n_components=10, solver="pcd", regularizer="squaredl12", beta=1e-3, gamma=1e-4,
          alpha=1e-3, max_iter=3, tol=-1.0, random_state=0, mean=True)),
    ("C2s", dict(n=20000, d=2000, r=50, seed=1, kernel="anova", degree=3, clf=True),
     dict(degree=3, loss="logistic", n_components=8, solver="pcd", regularizer="omegati", beta=1e-4,
          gamma=1e-5, alpha=1e-4, max_iter=2, tol=-1.0, random_state=0, mean=True)),
    ("C3s", dict(n=20000, d=2000, r=50, seed=2, kernel="anova", degree=2, clf=False),
     dict(degree=2, n_components=32, solver="pbcd", regularizer="omegacs", beta=1e-4, gamma=1e-5,
          alpha=1e-4, max_iter=2, tol=-1.0, random_state=0, mean=True)),
    ("C5s", dict(n=20000, d=5000, r=39, seed=4, kernel="anova", degree=2, clf=True),
     dict(degree=2, loss="logistic", n_components=32, solver="psgd", regularizer="squaredl12",
          alpha=1e-5, beta=1e-5, gamma=1e-4, max_iter=2, tol=-1.0, random_state=0, eta0=0.1,
          n_iter_no_change=10 ** 9)),
]


@pytest.mark.parametrize("tag,prob,kw", CASES_ORACLE, ids=[c[0] for c in CASES_ORACLE])
def test_scaled_baseline_configs_match_oracle(tag, prob, kw):
    X, y = _problem(**prob)
    est, out, frac = _compare_fm(kw, X, y, TOL)   # (psgd: the planned path sums in fixed order -- 1e-9 like the rest)
    print(tag, "nonzero fraction of P_", frac)


def test_all_subsets_c4_scaled_matches_oracle():
    import sparsepoly_b200 as S
    from oracle import oracle as O
    X, y = _problem(n=20000, d=800, r=20, seed=3, kernel="all", degree=2, clf=True)
    kw = dict(loss="squared_hinge", n_components=8, solver="pcd", regularizer="omegati", beta=1e-4,
              gamma=1e-5, mean=True, max_iter=2, tol=-1.0, random_state=0)
    est = _fit(S.SparseAllSubsetsClassifier(**kw), X, y)
    out = O.fit_all_subsets(X, y, **kw)
    assert rel_err(est.P_, out["P_"]) <= TOL
    assert same_support(est.P_, out["P_"])
    _check_objective(est, X, y, out["P_"], None)


@pytest.mark.parametrize("d,k", [(1, 1), (37, 3), (500, 16), (5000, 32), (3000, 100), (100000, 8), (0, 4)])
def test_reg_eval_kernels_match_oracle(d, k):
    """sp_reg_eval (objective.cu) for every regularizer x degree against the oracle's sequential
    folds; tree-ordered sums of non-negative terms: 1e-12."""
    import torch
    from sparsepoly_b200 import solvers
    from oracle import oracle as O
    rng = np.random.RandomState(d + k)
    scale = 0.5 / max(d, 1) ** 0.5                      # keeps prod_j (1 + |p_j|) finite
    P_dk = scale * rng.randn(d, k) * (rng.rand(d, k) < 0.6)
    P_dev = torch.from_numpy(P_dk).cuda()
    P_kd = np.ascontiguousarray(P_dk.T)
    for reg in ("l1", "l21", "squaredl12", "squaredl21"):
        got = solvers.reg_eval(P_dev, reg, 2).item()
        want = O.reg_eval(P_kd, reg, 2)
        assert abs(got - want) <= 1e-12 * max(abs(want), 1e-300), (reg, got, want)
    for reg in ("omegati", "omegacs"):
        for degree in (1, 2, 3, 4, 5, -1):
            got = solvers.reg_eval(P_dev, reg, degree).item()
            want = O.reg_eval(P_kd, reg, degree)
            assert abs(got - want) <= 1e-12 * max(abs(want), 1e-300), (reg, degree, got, want)
    with pytest.raises(ValueError):
        solvers.reg_eval(P_dev, "omegati", 9)


@pytest.mark.parametrize("loss", ["squared", "logistic", "squared_hinge"])
def test_loss_sum_and_sqnorm_match_oracle(loss):
    import torch
    from sparsepoly_b200 import solvers
    from oracle import oracle as O
    rng = np.random.RandomState(3)
    for n in (1, 1000, 300001):
        p = 8.0 * rng.randn(n)
        y = np.where(rng.rand(n) < 0.5, -1.0, 1.0)
        rec = np.zeros((n, 4))
        rec[:, 0], rec[:, 1] = p, y
        rec_dev = torch.from_numpy(rec).cuda().reshape(-1)
        got = solvers.loss_sum(rec_dev, rec_dev[1:], loss, n, pred_stride=4, y_stride=4).item()
        want = O.loss_sum(p, y, loss)
        assert abs(got - want) <= 1e-12 * abs(want)
        assert abs(solvers.sqnorm(torch.from_numpy(p).cuda()).item() - float(np.dot(p, p))) <= 1e-12 * np.dot(p, p)


def test_predict_matches_oracle_and_kernels_module():
    from sparsepoly_b200 import kernels, synth
    from oracle import oracle as O
    X = synth.uniform_sparse(3000, 400, 30, 7)
    rng = np.random.RandomState(0)
    P = 0.3 * rng.randn(7, 400)
    lams = np.sign(rng.randn(7))
    for deg in (2, 3, 4, 5):
        K = kernels.anova_kernel(X, P, deg)
        Kd = O.kernel_rows_dp(X, np.ascontiguousarray(P.T), deg)
        assert rel_err(K, Kd) <= 1e-13
        assert rel_err(kernels.poly_predict(X, P, lams, "anova", deg),
                       O.poly_predict(X, P, lams, "anova", deg)) <= 1e-9
    assert rel_err(kernels.all_subsets_kernel(X, 0.2 * P), O.all_subsets_kernel(X, 0.2 * P)) <= 1e-13
    # empty rows / empty matrix edge cases
    Xe = sp.csr_matrix((5, 400))
    assert np.array_equal(kernels.anova_kernel(Xe, P, 2), np.zeros((5, 7)))
    assert np.array_equal(kernels.all_subsets_kernel(Xe, P), np.ones((5, 7)))


@pytest.mark.parametrize("sweep", ["cluster", "window"])
def test_ragged_and_dense_columns(sweep, monkeypatch):
    """empty columns, one dense column (slice longer than a CTA: slow path), 1-sample data."""
    import sparsepoly_b200 as S
    monkeypatch.setenv("SPARSEPOLY_B200_SWEEP", sweep)
    from oracle import oracle as O
    rng = np.random.RandomState(3)
    n, d = 700, 9
    M = sp.random(n, d, density=0.05, format="lil", random_state=rng, data_rvs=rng.randn)
    M[:, 4] = rng.randn(n, 1)          # dense column
    M[:, 2] = 0                        # empty column
    X = sp.csr_matrix(M)
    y = rng.randn(n)
    for solver, reg in (("pcd", "l1"), ("pcd", "omegati"), ("pbcd", "omegacs"), ("pbcd", "l21")):
        kw = dict(degree=3, n_components=3, solver=solver, regularizer=reg, beta=0.1, gamma=0.01,
                  alpha=0.1, max_iter=3, tol=-1.0, random_state=1, fit_lower="explicit")
        est = _fit(S.SparseFactorizationMachineRegressor(**kw), X, y)
        out = O.fit_fm(X, y, loss="squared", **kw)
        assert rel_err(est.P_, out["P_"]) <= TOL, (solver, reg)
        assert rel_err(est.w_, out["w_"]) <= TOL
        assert same_support(est.P_, out["P_"])


def test_prox_operators_match_reference_vectors():
    import torch
    from golden_util import GOLD
    from sparsepoly_b200 import solvers
    z = np.load(os.path.join(GOLD, "reference_prox.npz"))
    for reg in ("l1", "l21", "squaredl12", "squaredl21"):
        for t in range(4):
            P = torch.from_numpy(np.ascontiguousarray(z[f"in_{t}"])).cuda()
            work = solvers.prox_work(P.shape[0], P.shape[1], P.device)
            solvers.prox(P, reg, float(z[f"strength_{t}"]), work)
            got, want = P.cpu().numpy(), z[f"{reg}_{t}"]
            assert rel_err(got, want) <= 1e-12, (reg, t)
            assert np.array_equal(got != 0, want != 0), (reg, t)


def test_squaredl12_prox_large_columns_vs_oracle():
    """prox over d=200k rows x 32 columns (C5-shaped column length / 5): same theta, S."""
    import torch
    from oracle import oracle as O
    from sparsepoly_b200 import solvers
    rng = np.random.RandomState(11)
    P = rng.randn(200000, 32) * (rng.rand(200000, 32) < 0.3)
    for strength in (1e-6, 1e-4):
        Pd = torch.from_numpy(P.copy()).cuda()
        solvers.prox(Pd, "squaredl12", strength, solvers.prox_work(*P.shape, Pd.device))
        Q = P.copy()
        O.Reg("squaredl12", *P.shape).prox(Q, strength)
        got = Pd.cpu().numpy()
        assert rel_err(got, Q) <= 1e-12
        assert np.array_equal(got != 0, Q != 0)
        assert np.all(np.abs(got) <= np.abs(P))          # magnitudes never grow (test_prox.py:70-76)


def test_callback_verbose_and_warm_start(capsys):
    import sparsepoly_b200 as S
    rec, X, arr = load_case("pcd_fm_sql12_squared")
    seen = []
    kw = dict(rec["kw"], max_iter=3, verbose=True, n_calls=1,
              callback=lambda est: seen.append(est.P_.copy()) or None)
    est = _fit(S.SparseFactorizationMachineRegressor(**kw), X, arr["y"])
    out = capsys.readouterr().out
    assert "Iteration 1 violation sum" in out and len(seen) == 3
    assert np.array_equal(seen[-1], est.P_)
    # warm start continues from the stored solution
    est.set_params(warm_start=True, max_iter=1, callback=None, verbose=False)
    P_before = est.P_.copy()
    _fit(est, X, arr["y"])
    assert not np.array_equal(P_before, est.P_)
    with pytest.raises(Exception):
        S.SparseFactorizationMachineRegressor().predict(X)


def test_device_csc_transpose_matches_scipy():
    """DeviceDataset builds the CSC copy on the device (stable sort by column): bit-identical to scipy."""
    import torch
    from sparsepoly_b200 import synth
    from sparsepoly_b200.dataset import DeviceDataset
    X = synth.uniform_sparse(5000, 700, 13, 21)
    X[17] = 0                                     # an empty row; column 3 emptied below
    X = sp.csr_matrix(X)
    X[:, 3] = 0
    X.eliminate_zeros()
    ds = DeviceDataset(X, need_csr=True, need_csc=True)
    Xc = sp.csc_matrix(X)
    Xc.sort_indices()
    ip, ix, dt = (t.cpu().numpy() for t in ds.csc)
    assert np.array_equal(ip, Xc.indptr) and np.array_equal(ix, Xc.indices) and np.array_equal(dt, Xc.data)


@pytest.mark.parametrize("name", large_case_names())
def test_matches_reference_beyond_toy_sizes(name):
    """CUDA backend against the UNMODIFIED reference at C1 full size (5 and 25 epochs), C2/50, C3/50, C4/10, two
    Criteo-shaped psgd problems and the omegacs negative-dcache fixture (tests/golden/reference_large/)."""
    rec, X, arr = load_large_case(name)
    est = _fit(_estimator(rec), X, arr["y"])
    assert rel_err(est.P_, arr["P_"]) <= TOL
    assert same_support(est.P_, arr["P_"])
    if "w_" in arr:
        assert rel_err(est.w_, arr["w_"]) <= TOL
    assert est.n_iter_ == int(arr["n_iter_"])
    if "it_" in arr:
        assert est.it_ == int(arr["it_"])
    pred = est.decision_function(arr["Xte"]) if rec["clf"] else est.predict(arr["Xte"])
    assert rel_err(pred, arr["pred_te"]) <= TOL
    _check_objective(est, X, arr["y"], arr["P_"], arr.get("w_"))


PSGD_PLANNED = [
    # Criteo-shaped inputs: 13 dense columns (split over many chunks of the column pass) + Zipf tails
    ("sql12_auto", dict(degree=2, loss="logistic", n_components=32, regularizer="squaredl12", alpha=1e-5, beta=1e-5,
                        gamma=1e-4, eta0=0.1, max_iter=3)),
    ("sql12_k16_batch1000_shuffle", dict(degree=2, loss="squared_hinge", n_components=16, regularizer="squaredl12",
                                         alpha=1e-4, beta=1e-4, gamma=3e-4, eta0=0.05, max_iter=2, batch_size=1000,
                                         shuffle=True, learning_rate="invscaling", power_t=0.3)),
    ("l1_deg3_explicit_k40", dict(degree=3, loss="logistic", n_components=40, regularizer="l1", alpha=1e-5, beta=1e-5,
                                  gamma=2e-5, eta0=0.1, max_iter=2, fit_lower="explicit", batch_size=3000)),
    ("sql12_deg4_nolinear_k5", dict(degree=4, loss="squared", n_components=5, regularizer="squaredl12", alpha=1e-4,
                                    beta=1e-3, gamma=1e-4, eta0=0.02, max_iter=2, fit_lower=None, fit_linear=False,
                                    batch_size=20000, learning_rate="constant")),
    ("l1_k100_one_batch", dict(degree=2, loss="logistic", n_components=100, regularizer="l1", alpha=1e-5, beta=1e-5,
                               gamma=1e-5, eta0=0.1, max_iter=3, batch_size=10 ** 6)),
]


@pytest.mark.parametrize("tag,kw", PSGD_PLANNED, ids=[c[0] for c in PSGD_PLANNED])
def test_psgd_planned_path_matches_oracle(tag, kw):
    """planned path (psgd_plan.cu: rows / cols / split / stats / solve kernels) against the oracle's psgd."""
    import sparsepoly_b200 as S
    from oracle import oracle as O
    from sparsepoly_b200 import synth
    X = synth.criteo_like(20000, 4000, 4)
    rng = np.random.RandomState(1)
    clf = kw["loss"] != "squared"
    y = np.where(rng.rand(20000) < 0.3, 1.0, -1.0) if clf else rng.randn(20000)
    kw = dict(kw, solver="psgd", tol=-1.0, random_state=0, n_iter_no_change=10 ** 9)
    ekw = dict(kw)
    cls = S.SparseFactorizationMachineClassifier if clf else S.SparseFactorizationMachineRegressor
    if not clf:
        ekw.pop("loss")
    est = _fit(cls(**ekw), X, y)
    out = O.fit_fm(X, y, **kw)
    assert rel_err(est.P_, out["P_"]) <= TOL
    assert same_support(est.P_, out["P_"])
    assert rel_err(est.w_, out["w_"]) <= TOL
    assert est.it_ == out["it_"]
    frac = float(np.mean(out["P_"] != 0))
    print(tag, "nonzero fraction of P_", frac, est._psgd_stats)
    # bit-reproducible run to run (fixed summation order everywhere; the reference is deterministic too)
    est2 = _fit(cls(**ekw), X, y)
    assert np.array_equal(est.P_, est2.P_) and np.array_equal(est.w_, est2.w_)


def test_psgd_planned_and_dense_gradient_paths_agree(monkeypatch):
    """l1 / squaredl12 through the dense-gradient path (psgd.cu: atomics, dense step, whole-matrix prox) vs the
    planned path: same model to rounding."""
    import sparsepoly_b200 as S
    from sparsepoly_b200 import solvers, synth
    X = synth.criteo_like(8000, 2500, 9)
    y = np.where(np.random.RandomState(2).rand(8000) < 0.3, 1.0, -1.0)
    for reg in ("squaredl12", "l1"):
        kw = dict(degree=2, loss="logistic", n_components=8, solver="psgd", regularizer=reg, alpha=1e-4, beta=1e-4,
                  gamma=1e-3 if reg == "squaredl12" else 1e-4, eta0=0.1, max_iter=2, tol=-1.0, random_state=0,
                  n_iter_no_change=10 ** 9, batch_size=700)
        a = _fit(S.SparseFactorizationMachineClassifier(**kw), X, y)
        monkeypatch.setattr(solvers, "PLANNED_REGS", ())
        b = _fit(S.SparseFactorizationMachineClassifier(**kw), X, y)
        monkeypatch.undo()
        assert rel_err(a.P_, b.P_) <= 1e-10 and rel_err(a.w_, b.w_) <= 1e-10, reg
        assert same_support(a.P_, b.P_)


def test_psgd_callback_sees_current_model_and_lazy_frame_survives():
    """callback(self) every epoch forces the lazily scaled storage back into the model mid-fit; the fit must be
    unaffected (same result as without a callback)."""
    import sparsepoly_b200 as S
    from sparsepoly_b200 import synth
    X = synth.criteo_like(6000, 1500, 3)
    y = np.where(np.random.RandomState(4).rand(6000) < 0.3, 1.0, -1.0)
    kw = dict(degree=2, loss="logistic", n_components=8, solver="psgd", regularizer="squaredl12", alpha=1e-4, beta=1e-2,
              gamma=1e-3, eta0=0.3, max_iter=4, tol=-1.0, random_state=0, n_iter_no_change=10 ** 9, batch_size=500,
              learning_rate="constant")
    seen = []
    a = _fit(S.SparseFactorizationMachineClassifier(callback=lambda e: seen.append(e.P_.copy()) or None, n_calls=1, **kw), X, y)
    b = _fit(S.SparseFactorizationMachineClassifier(**kw), X, y)
    assert len(seen) == 4 and np.array_equal(seen[-1], a.P_)
    assert rel_err(a.P_, b.P_) <= 1e-12 and same_support(a.P_, b.P_)


# ------------------------------------------------------------------ sharded psgd: 2 processes, peer memory (CUDA IPC)
def _sharded_worker(rank, world, port, out_dir, n_dev):
    import sys
    import torch
    import torch.distributed as dist
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, root)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank % n_dev)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    import sparsepoly_b200 as S
    from sparsepoly_b200 import distributed, synth
    distributed.enable_sharding()
    res = {}
    for tag, kw in _SHARDED_CASES:
        X = synth.criteo_like(_SH_N, _SH_D, 21 + rank)
        y = np.where(np.random.RandomState(31 + rank).rand(_SH_N) < 0.3, 1.0, -1.0)
        est = S.SparseFactorizationMachineClassifier(random_state=rank, **kw)    # different draws: rank 0's must win
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            est.fit(X, y)
        res[tag + "/P"], res[tag + "/w"], res[tag + "/it"] = est.P_, est.w_, np.array(est.it_)
        Xte = synth.criteo_like(50 + 10 * rank, _SH_D, 77 + rank)
        res[tag + "/pred"] = distributed.sharded_predict(est, Xte)
    np.savez(os.path.join(out_dir, f"rank{rank}.npz"), **res)
    dist.barrier()
    dist.destroy_process_group()


_SH_N, _SH_D = 3000, 1200
_SHARDED_CASES = [
    ("sql12", dict(degree=2, loss="logistic", n_components=8, solver="psgd", regularizer="squaredl12", alpha=1e-4,
                   beta=1e-4, gamma=1e-3, eta0=0.1, max_iter=2, tol=-1.0, n_iter_no_change=10 ** 9, batch_size=512)),
    ("l1_deg3", dict(degree=3, loss="logistic", n_components=4, solver="psgd", regularizer="l1", alpha=1e-4,
                     beta=1e-4, gamma=1e-4, eta0=0.1, max_iter=2, tol=-1.0, n_iter_no_change=10 ** 9, batch_size=1000,
                     fit_lower="explicit")),
]


def test_sharded_psgd_two_ranks_matches_oracle(tmp_path):
    """Two ranks (one process and one GPU each), samples
    sharded, P sharded by rows in peer memory: pull / push / owner / statistics exchange of psgd_plan.cu against the
    oracle on the interleaved data set (reference optimizer/psgd.py:150-198), 1e-9; batch prediction sharded too."""
    import torch
    import torch.multiprocessing as mp
    from oracle import oracle as O
    from sparsepoly_b200 import synth
    from sparsepoly_b200.distributed import interleave_shards
    world = 2
    if torch.cuda.device_count() < world:
        # kernels of different ranks wait on one another through peer-memory flags; on ONE device nothing
        # guarantees they are co-scheduled (B200_PROFILING.md: Xid 109).  profiles/r02_* hold the 2-GPU logs.
        pytest.skip("needs one GPU per rank")
    port = 33500 + (os.getpid() % 2000)
    mp.spawn(_sharded_worker, args=(world, port, str(tmp_path), torch.cuda.device_count()), nprocs=world, join=True)
    z = [np.load(tmp_path / f"rank{r}.npz") for r in range(world)]
    Xs = [synth.criteo_like(_SH_N, _SH_D, 21 + r) for r in range(world)]
    ys = [np.where(np.random.RandomState(31 + r).rand(_SH_N) < 0.3, 1.0, -1.0) for r in range(world)]
    for tag, kw in _SHARDED_CASES:
        b_loc = kw["batch_size"] // world
        order = interleave_shards([np.arange(_SH_N) + r * _SH_N for r in range(world)], b_loc * world)
        Xall, yall = sp.vstack(Xs).tocsr()[order], np.concatenate(ys)[order]
        out = O.fit_fm(Xall, yall, random_state=0, **dict(kw, batch_size=b_loc * world))
        for r in range(world):
            assert rel_err(z[r][tag + "/P"], out["P_"]) <= TOL, (tag, r)
            assert same_support(z[r][tag + "/P"], out["P_"])
            assert rel_err(z[r][tag + "/w"], out["w_"]) <= TOL
            assert int(z[r][tag + "/it"]) == out["it_"]
        assert np.array_equal(z[0][tag + "/P"], z[1][tag + "/P"])             # replicas end identical
        Xte = sp.vstack([synth.criteo_like(50 + 10 * r, _SH_D, 77 + r) for r in range(world)]).tocsr()
        want = O.fm_output(Xte, out["P_"], out["w_"], out["lams_"], kw["degree"], True, kw.get("fit_lower", "explicit"))
        assert rel_err(z[0][tag + "/pred"], want) <= TOL and np.array_equal(z[0][tag + "/pred"], z[1][tag + "/pred"])


def test_transpose_handles_more_than_two_million_rows():
    """ADVICE r1: sp_transpose_f64 used grid.y for the row tiles (<= 65 535 tiles = 2.1 M rows); pbcd / psgd transpose
    P [d, k] at every sync, so a sparse CTR feature space of d > 2.1 M made fit() fail at its very end."""
    import torch
    from sparsepoly_b200 import solvers
    t = torch.arange(2_200_003 * 3, dtype=torch.float64, device="cuda").reshape(2_200_003, 3)
    out = solvers.transpose(t)
    assert out.shape == (3, 2_200_003) and torch.equal(out, t.t().contiguous())
    out2 = solvers.transpose(out)
    assert torch.equal(out2, t)
