"""The value each epoch's stopping rule compares, against the oracle, and fits that stop on it.

With the defaults (tol=1e-6, n_iter_no_change=5) the number of epochs, and so the model, depends on one value per
epoch: the violation sum of pcd / pbcd / all-subsets (accumulated inside the sweep kernels next to the update) and
psgd's mean epoch loss (summed by the planned path in fixed order, by the dense-gradient path with fp64 atomics,
over ranks by sharded psgd).  The coefficient parity tests run with tol=-1, where that value decides nothing.

  * trace parity (tol=-1): the device's per-epoch values, parsed from the verbose lines, against the oracle's
    out["trace"] on every path that computes them; each case asserts that it reached the path it names;
  * stops: tol / n_iter_no_change chosen from the oracle's trace (tests/test_stopping_cpu.py) so that device and
    oracle must stop at one chosen epoch with every decision a margin of >= 1e-6 away; n_iter_, it_, the convergence
    warning, P_ / w_ and the objective must then match the oracle's.

Bars: |v_dev - v_ref| <= 1e-9 max(v_ref, 1e-6 |coef_ref|_1) for violation sums (the floor covers late epochs whose
violation is a few ulps of large coefficients); 1e-12 relative for the planned path's losses, 1e-10 for the
dense-gradient path's (fp64 atomics in no fixed order)."""
import contextlib
import io
import math
import os
import warnings

import numpy as np
import pytest
import scipy.sparse as sp

import test_partial_fit_gpu as PF
from golden_util import load_large_case, rel_err, same_support
from test_kernel_variants_gpu import (PBCD_PROB, PBCD_WINDOW_PROB, PCD5_PROB, PROF_PSGD_GRAD, PROF_SWEEP_PBCD, PSGD_D,
                                      PSGD_N, _fm_estimator, _launches, _oracle, _pbcd_estimator, _pbcd_kw, _pcd5_kw,
                                      _pick_nz, _profile)
from test_parity_gpu import SPEC_CASES, WINDOW_ORACLE, _check_objective, _problem, _wspec_read
from test_stopping_cpu import (choose_plateau_tol, first_drop, parse_traces, replay_plateau, replay_viol, tol_never,
                               tol_stopping_at)

pytestmark = pytest.mark.gpu

TOL = 1e-9
LOSS_TOL = {"planned": 1e-12, "dense": 1e-10}
PROF_SWEEP_PCD = 2                      # kernel class of sp_profile_* (csrc/common.cuh)
NOT_CONVERGED = "Objective did not converge"


# ------------------------------------------------------------------------------------------------------ helpers
def _not_converged(caught):
    return sum(NOT_CONVERGED in str(w.message) for w in caught)


def trace_of(est, X, y, profile=False):
    """(trace, warned, launches): est fitted on (X, y) with verbose=True; the per-epoch values its stopping rule
    compared, parsed from the verbose lines; whether fit warned that the objective did not converge; and the kernel
    launch counts of sp_profile_* when profile=True."""
    est.set_params(verbose=True)
    buf = io.StringIO()
    if profile:
        _profile(True)
    try:
        with warnings.catch_warnings(record=True) as caught, contextlib.redirect_stdout(buf):
            warnings.simplefilter("always")
            est.fit(X, y)
        cnt = _launches() if profile else None
    finally:
        if profile:
            _profile(False)
    traces = parse_traces(buf.getvalue())
    assert len(traces) == 1, buf.getvalue()[:2000]
    warned = _not_converged(caught)
    assert warned <= 1
    return traces[0], bool(warned), cnt


def _coef_l1(out):
    return float(np.abs(out["P_"]).sum() + (np.abs(out["w_"]).sum() if "w_" in out else 0.0))


def check_viol_trace(tag, path, got, out, est=None):
    """Violation sums entry by entry against out["trace"]; prints the worst error as a fraction of the bar."""
    want = out["trace"]
    assert len(got) == len(want), (tag, got, want)
    floor = 1e-6 * _coef_l1(out)
    worst = 0.0
    for i, (g, w) in enumerate(zip(got, want)):
        bar = TOL * max(w, floor)
        assert abs(g - w) <= bar, (tag, i, g, w, bar)
        worst = max(worst, abs(g - w) / bar if bar > 0.0 else 0.0)
    bits = ""
    if est is not None and np.array_equal(est.P_, out["P_"]):
        bits = f"; P_ bit-identical, trace bit-identical: {list(got) == list(want)}"
    print(f"{tag} [{path}]: {len(got)} epochs, worst violation error {worst:.3g} of the bar{bits}")
    return worst


def check_loss_trace(tag, path, got, want, kind):
    assert len(got) == len(want), (tag, got, want)
    rel = LOSS_TOL[kind]
    worst = max(abs(g - w) / (rel * abs(w)) for g, w in zip(got, want))
    assert worst <= 1.0, (tag, got, want)
    print(f"{tag} [{path}]: {len(got)} epochs, worst loss error {worst:.3g} of {rel:g} relative, "
          f"bit-identical: {list(got) == list(want)}")
    return worst


def _with_env(monkeypatch, env):
    for k, v in env.items():
        monkeypatch.setenv(k, str(v))


def _fm_oracle(prob, kw):
    from oracle import oracle as O
    X, y = _problem(**prob)
    okw = dict(kw)
    okw.setdefault("loss", "squared")
    return X, y, _oracle(repr(("stop", sorted(prob.items()), sorted(okw.items(), key=str))),
                         lambda: O.fit_fm(X, y, **okw))


def _all_oracle(prob, kw):
    from oracle import oracle as O
    X, y = _problem(**prob)
    return X, y, _oracle(repr(("stop-all", sorted(prob.items()), sorted(kw.items(), key=str))),
                         lambda: O.fit_all_subsets(X, y, **kw))


def _all_estimator(kw):
    import sparsepoly_b200 as S
    if kw.get("loss", "squared") == "squared":
        return S.SparseAllSubsetsRegressor(**{k: v for k, v in kw.items() if k != "loss"})
    return S.SparseAllSubsetsClassifier(**kw)


# ============================================================================ 1. pcd: cluster sweep (pcd.cu)
PCD_PROB = dict(PCD5_PROB, clf=False)
PCD_CLF_PROB = dict(PCD5_PROB, clf=True)
_SQL12 = dict(degree=2, n_components=6, solver="pcd", regularizer="squaredl12", beta=1e-4, gamma=1e-6, alpha=1e-3,
              max_iter=4, tol=-1.0, random_state=0, mean=True)
_FM3 = dict(degree=3, loss="logistic", n_components=8, solver="pcd", regularizer="omegati", beta=1e-4, gamma=1e-5,
            alpha=1e-4, max_iter=3, tol=-1.0, random_state=0, mean=True, fit_lower="explicit")
PCD_CLUSTER = [
    # (tag, problem, kw, (n_cta, threads), NZ of pick_nz)
    ("deg2_nz1", PCD_PROB, _SQL12, (1, 256), 1),
    ("deg2_nz2", PCD_PROB, _SQL12, (2, 32), 2),
    ("deg5_nz1", PCD_CLF_PROB, _pcd5_kw("logistic", "omegati", "explicit"), (1, 256), 1),
    ("deg5_nz2", PCD_CLF_PROB, _pcd5_kw("logistic", "omegati", "explicit"), (2, 32), 2),
    ("deg3_explicit", PCD_CLF_PROB, _FM3, (4, 64), 1),
    ("no_linear_l1", PCD_PROB, dict(_SQL12, regularizer="l1", beta=1e-4, gamma=1e-5, fit_linear=False), (1, 256), 1),
    ("shuffle", PCD_PROB, dict(_SQL12, shuffle=True), (2, 32), 2),
]


@pytest.mark.parametrize("tag,prob,kw,geom,nz", PCD_CLUSTER, ids=[c[0] for c in PCD_CLUSTER])
def test_pcd_cluster_sweep_trace(tag, prob, kw, geom, nz, monkeypatch):
    _with_env(monkeypatch, dict(SPARSEPOLY_B200_SWEEP="cluster", SPARSEPOLY_B200_NCTA=geom[0],
                                SPARSEPOLY_B200_THREADS=geom[1]))
    X, y, out = _fm_oracle(prob, kw)
    est = _fm_estimator(kw)
    got, warned, _ = trace_of(est, X, y)
    plan, ds = est._dev_state["plan"], est._dev_state["ds"]
    assert plan.mode == "cluster" and (plan.n_cta, plan.threads) == geom
    assert _pick_nz(ds, plan.n_cta, plan.threads) == nz
    assert warned and rel_err(est.P_, out["P_"]) <= TOL and 0.01 < np.mean(out["P_"] != 0) < 0.99
    check_viol_trace(tag, f"pcd cluster sweep NCTA={geom[0]} threads={geom[1]} NZ={nz}", got, out, est)


# ============================================================================ 2. pcd: window sweep (pcd_window.cu)
WINDOW_PROB = dict(n=100000, d=5000, r=10, seed=5, kernel="anova")
_FM3_WINDOW = dict(WINDOW_ORACLE[0][4])


@pytest.mark.parametrize("horizon,near", [(0, 1), (1, 2)])
def test_pcd_window_sweep_trace(horizon, near, monkeypatch):
    _with_env(monkeypatch, dict(SPARSEPOLY_B200_SWEEP="window", SPARSEPOLY_B200_HORIZON=horizon,
                                SPARSEPOLY_B200_NEAR=near))
    X, y, out = _fm_oracle(dict(WINDOW_PROB, degree=3, clf=True), _FM3_WINDOW)
    est = _fm_estimator(_FM3_WINDOW)
    got, warned, _ = trace_of(est, X, y)
    stats = est._dev_state["plan"].wplan.stats
    assert est._dev_state["plan"].mode == "window" and (stats["horizon"], stats["near"]) == (horizon, near), stats
    assert warned and rel_err(est.P_, out["P_"]) <= TOL
    check_viol_trace("fm3_omegati_logistic", f"pcd window sweep horizon={horizon} near={near}", got, out, est)


SPEC_TRACE = [c for c in SPEC_CASES if c[0] != "l1_all_zero"]
_REJECTED = {}


@pytest.mark.parametrize("tag,degree,clf,kw", SPEC_TRACE, ids=[c[0] for c in SPEC_TRACE])
def test_speculative_window_trace(tag, degree, clf, kw, monkeypatch):
    """Zero-update speculation: the chain warp commits a run of positions up to the first mover and adds that
    mover's |update| to the violation once; rejected positions are redone.  With and without speculation the
    trace must match the oracle's, and each other's."""
    monkeypatch.setenv("SPARSEPOLY_B200_SWEEP", "window")
    X, y, out = _fm_oracle(dict(WINDOW_PROB, degree=degree, clf=clf), kw)
    _wspec_read()
    est = _fm_estimator(kw)
    got, _, _ = trace_of(est, X, y)
    n_spec, n_rej = _wspec_read()
    assert est._dev_state["plan"].mode == "window"
    assert n_spec > 0, "speculation never engaged"
    _REJECTED[tag] = n_rej
    check_viol_trace(tag, f"pcd window sweep, speculation: {n_spec} positions, {n_rej} rejected", got, out, est)
    monkeypatch.setenv("SPARSEPOLY_B200_SPEC", "0")
    est0 = _fm_estimator(kw)
    got0, _, _ = trace_of(est0, X, y)
    assert _wspec_read() == (0, 0)
    check_viol_trace(tag, "pcd window sweep, SPARSEPOLY_B200_SPEC=0", got0, out, est0)
    floor = 1e-6 * _coef_l1(out)
    for a, b in zip(got, got0):
        assert abs(a - b) <= TOL * max(b, floor), (got, got0)
    print(tag, "speculative and in-order traces bit-identical:", got == got0)


def test_speculative_window_trace_saw_rejections():
    """At least one speculation regime above redid a position (the rejection branch fed the trace)."""
    if len(_REJECTED) < len(SPEC_TRACE):
        pytest.skip("needs every test_speculative_window_trace case in this run")
    assert max(_REJECTED.values()) > 0, _REJECTED


def test_dead_component_shortcut_trace(monkeypatch):
    """l1_all_zero: every component is zero after the first epoch, so sp_pcd_epoch skips their sweeps and later
    violations come from the linear sweep alone.  One sweep launch per component in epoch 0 and one linear sweep
    per epoch."""
    from oracle import oracle as O
    tag, degree, clf, kw = next(c for c in SPEC_CASES if c[0] == "l1_all_zero")
    monkeypatch.setenv("SPARSEPOLY_B200_SWEEP", "window")
    X, y, out = _fm_oracle(dict(WINDOW_PROB, degree=degree, clf=clf), kw)
    first = _oracle(repr(("l1_all_zero", 1)), lambda: O.fit_fm(X, y, **dict(kw, max_iter=1, loss="squared")))
    assert not np.any(first["P_"]) and not np.any(out["P_"])
    est = _fm_estimator(kw)
    got, _, cnt = trace_of(est, X, y, profile=True)
    assert est._dev_state["plan"].mode == "window"
    assert cnt[PROF_SWEEP_PCD] == kw["max_iter"] + kw["n_components"], cnt
    check_viol_trace(tag, "dead-component shortcut, linear sweep only after epoch 0", got, out, est)


# ============================================================================ 3. pbcd (pbcd.cu, pbcd_window.cu)
PBCD_CASES = [
    # (tag, problem, kw, degree, sweep)
    ("k5_deg5_omegacs_window", PBCD_WINDOW_PROB, _pbcd_kw(5, 5, "omegacs", gamma=1e-7, max_iter=3), 5, "window"),
    ("k32_deg5_l21_window", PBCD_WINDOW_PROB, _pbcd_kw(32, 5, "l21", gamma=1e-5, max_iter=3), 5, "window"),
    ("k5_deg3_omegacs_cluster", PBCD_PROB, _pbcd_kw(5, 3, "omegacs", max_iter=4), 3, "cluster"),
    ("k32_sql21_cluster", PBCD_PROB, _pbcd_kw(32, 2, "squaredl21", max_iter=4), 2, "cluster"),
    ("k33_l21_kch2", PBCD_PROB, _pbcd_kw(33, 3, "l21", max_iter=3), 3, "cluster"),
    ("k64_omegacs_kch2", PBCD_PROB, _pbcd_kw(64, 2, "omegacs", max_iter=3), 2, "cluster"),
    ("k100_sql21_kch4", PBCD_PROB, _pbcd_kw(100, 2, "squaredl21", max_iter=3), 2, "cluster"),
    ("k128_l21_kch4", PBCD_PROB, _pbcd_kw(128, 2, "l21", max_iter=3), 2, "cluster"),
]


@pytest.mark.parametrize("tag,prob,kw,degree,sweep", PBCD_CASES, ids=[c[0] for c in PBCD_CASES])
def test_pbcd_sweep_trace(tag, prob, kw, degree, sweep, monkeypatch):
    monkeypatch.setenv("SPARSEPOLY_B200_SWEEP", sweep)
    X, y, out = _fm_oracle(prob, kw)
    est = _pbcd_estimator(kw, degree)
    got, warned, cnt = trace_of(est, X, y, profile=True)
    plan = est._dev_state["plan"]
    assert plan.mode == sweep
    assert cnt[PROF_SWEEP_PBCD] == kw["max_iter"] * (degree - 1), cnt
    assert warned and rel_err(est.P_, out["P_"]) <= TOL and same_support(est.P_, out["P_"])
    check_viol_trace(tag, f"pbcd {sweep} sweep k={kw['n_components']} KCH={-(-kw['n_components'] // 32)}", got, out,
                     est)


@pytest.mark.parametrize("sweep", ["cluster", "window"])
def test_pbcd_omegacs_negative_dcache_trace(sweep, monkeypatch):
    """The omegacs_negative_dcache inputs, which enter the reference's negative-dcache recovery (omegacs.py:90-96)."""
    from oracle import oracle as O
    monkeypatch.setenv("SPARSEPOLY_B200_SWEEP", sweep)
    rec, X, arr = load_large_case("omegacs_negative_dcache")
    kw = dict(rec["kw"])
    O.branch_counts(reset=True)
    out = O.fit_fm(X, arr["y"], loss="squared", **kw)
    assert O.branch_counts()[0] >= 1, "the inputs no longer enter the negative-dcache branch"
    est = _pbcd_estimator(kw, kw["degree"])
    got, _, _ = trace_of(est, X, arr["y"])
    assert est._dev_state["plan"].mode == sweep
    check_viol_trace("omegacs_negative_dcache", f"pbcd {sweep} sweep, omegacs negative dcache", got, out, est)


# ============================================================================ 4. all-subsets
ALL_PROB = dict(n=20000, d=800, r=20, seed=3, kernel="all", degree=2)
ALL_CASES = [
    ("pcd_reg", False, dict(n_components=8, solver="pcd", regularizer="omegati", beta=1e-4, gamma=1e-5)),
    ("pcd_clf", True, dict(loss="squared_hinge", n_components=8, solver="pcd", regularizer="omegati", beta=1e-4,
                           gamma=1e-5)),
    ("pbcd_reg", False, dict(n_components=8, solver="pbcd", regularizer="omegacs", beta=1e-4, gamma=1e-6)),
    ("pbcd_clf", True, dict(loss="logistic", n_components=8, solver="pbcd", regularizer="l21", beta=1e-4,
                            gamma=1e-2)),
]


@pytest.mark.parametrize("tag,clf,kw", ALL_CASES, ids=[c[0] for c in ALL_CASES])
def test_all_subsets_trace(tag, clf, kw):
    kw = dict(kw, mean=True, max_iter=3, tol=-1.0, random_state=0)
    X, y, out = _all_oracle(dict(ALL_PROB, clf=clf), dict(kw, loss=kw.get("loss", "squared")))
    est = _all_estimator(kw)
    got, warned, _ = trace_of(est, X, y)
    assert warned and rel_err(est.P_, out["P_"]) <= TOL and 0.01 < np.mean(out["P_"] != 0) < 0.99
    check_viol_trace(tag, f"all-subsets {kw['solver']} {est._dev_state['plan'].mode} sweep", got, out, est)


# ============================================================================ 5. psgd
def _psgd_problem(seed=3, n=PSGD_N, d=PSGD_D):
    from sparsepoly_b200 import synth
    X = synth.criteo_like(n, d, seed)
    y = np.where(np.random.RandomState(seed + 1).rand(n) < 0.3, 1.0, -1.0)
    return X, y


def _psgd_kw(reg, k, **extra):
    kw = dict(degree=2, loss="logistic", n_components=k, solver="psgd", regularizer=reg, alpha=1e-4, beta=1e-4,
              gamma={"l1": 2e-4, "squaredl12": 1e-3, "l21": 1e-3, "squaredl21": 3e-4}[reg], eta0=0.1, max_iter=4,
              tol=-1.0, random_state=0, n_iter_no_change=10 ** 9, batch_size=2000, fit_lower="explicit")
    kw.update(extra)
    return kw


def _psgd_oracle(kw, seed=3):
    from oracle import oracle as O
    X, y = _psgd_problem(seed)
    return X, y, _oracle(repr(("stop-psgd", seed, sorted(kw.items(), key=str))), lambda: O.fit_fm(X, y, **kw))


PSGD_PLANNED = [
    ("l1_logistic_partial_batch", _psgd_kw("l1", 8, batch_size=3000)),
    ("l1_squared_hinge", _psgd_kw("l1", 16, loss="squared_hinge")),
    ("sql12_squared", _psgd_kw("squaredl12", 8, loss="squared", eta0=0.02)),
    ("sql12_logistic_shuffle_partial", _psgd_kw("squaredl12", 32, shuffle=True, batch_size=1500)),
    ("sql12_squared_hinge_deg3", _psgd_kw("squaredl12", 8, loss="squared_hinge", degree=3, batch_size=2500)),
]
PSGD_DENSE = [
    ("l21_k16_hot_tiles", _psgd_kw("l21", 16)),
    ("sql21_k32_hot_tiles", _psgd_kw("squaredl21", 32, batch_size=3000)),
    ("l21_k64", _psgd_kw("l21", 64, loss="squared_hinge")),
]


@pytest.mark.parametrize("tag,kw", PSGD_PLANNED + PSGD_DENSE, ids=[c[0] for c in PSGD_PLANNED + PSGD_DENSE])
def test_psgd_epoch_loss_trace(tag, kw):
    from sparsepoly_b200.dataset import DeviceDataset
    X, y, out = _psgd_oracle(kw)
    est = _fm_estimator(kw)
    got, warned, cnt = trace_of(est, X, y, profile=True)
    planned = kw["regularizer"] in ("l1", "squaredl12")
    assert ("plan_bytes" in est._psgd_stats) == planned, est._psgd_stats
    n_mb = math.ceil(PSGD_N / kw["batch_size"])
    if not planned:
        assert cnt[PROF_PSGD_GRAD] == kw["max_iter"] * n_mb, cnt
        if kw["n_components"] <= 32:          # KCH * NORD == 1: the hot-feature pre-reduction runs
            assert DeviceDataset(X, need_csr=True, need_csc=False).struct.n_hot_feat >= 13
    assert warned and est.it_ == out["it_"] and rel_err(est.P_, out["P_"]) <= TOL
    path = "planned" if planned else "dense"
    check_loss_trace(tag, f"psgd {path} path, {n_mb} minibatches, last {PSGD_N - (n_mb - 1) * kw['batch_size']} rows",
                     got, out["trace"], path)


def _zero_loss_problem(B):
    """Criteo-shaped rows plus two indicator columns set on the first two minibatches only: +1 rows carry the
    first, -1 rows the second.  With w = +-20 there, every margin of those minibatches is >= 1, so their
    squared-hinge losses, and every partial sum of them, are exactly 0.0."""
    X, y = _psgd_problem(seed=5)
    n, d = X.shape
    ind = np.zeros((n, 2))
    rows = np.arange(2 * B)
    ind[rows, np.where(y[rows] > 0, 0, 1)] = 1.0
    X = sp.hstack([X, sp.csr_matrix(ind)]).tocsr()
    w0 = np.zeros(d + 2)
    w0[d], w0[d + 1] = 20.0, -20.0
    P0 = 0.01 * np.random.RandomState(0).randn(1, 8, d + 2)
    return X, y, P0, w0


@pytest.mark.parametrize("reg", ["l1", "l21"])
def test_psgd_zero_loss_minibatches_trace(reg):
    """Minibatches whose loss sums to exactly 0.0 (the dense path skips adding such a group's sum)."""
    from oracle import oracle as O
    B = 2000
    X, y, P0, w0 = _zero_loss_problem(B)
    kw = _psgd_kw(reg, 8, loss="squared_hinge", max_iter=3, batch_size=B)
    margins = y * O.fm_output(X, P0, w0, np.ones(8), 2, True, "explicit")
    assert np.all(margins[:2 * B] >= 1.0) and np.mean(margins[2 * B:] >= 1.0) < 0.1
    out = O.fit_fm(X, y, P_init=P0, w_init=w0, **kw)
    est = _fm_estimator(dict(kw, warm_start=True))
    est.P_, est.w_ = P0.copy(), w0.copy()
    got, _, _ = trace_of(est, X, y)
    planned = reg == "l1"
    assert ("plan_bytes" in est._psgd_stats) == planned
    assert est.it_ == out["it_"] and rel_err(est.P_, out["P_"]) <= TOL
    path = "planned" if planned else "dense"
    check_loss_trace(f"zero_loss_{reg}", f"psgd {path} path, minibatches 0-1 with loss 0.0", got, out["trace"], path)


@pytest.mark.parametrize("reg", ["l1", "squaredl12", "l21", "squaredl21"])
def test_partial_fit_call_losses_match_oracle_call_by_call(reg):
    """The mean loss each partial_fit call reports ("Call i loss v"), against the oracle driven call by call."""
    sizes = [250, 130, 400, 77]
    X, y = PF._problem(sum(sizes), 700, 5, True)
    kw = PF._kw(reg, 2, 8, True, batch_size=100)
    est = PF._clf_est(dict(kw, verbose=True))
    want = []
    P = w = lams = None
    it = 1
    from oracle import oracle as O
    okw = {k: v for k, v in kw.items() if k not in ("solver", "tol", "n_iter_no_change", "max_iter")}
    buf = io.StringIO()
    for a, b in PF._bounds(sizes):
        out = O.fit_fm(X[a:b], y[a:b], solver="psgd", max_iter=1, tol=-1.0, n_iter_no_change=10 ** 9, P_init=P,
                       w_init=w, lams_init=lams, it_init=it, **okw)
        P, w, lams, it = out["P_"], out["w_"], out["lams_"], out["it_"]
        want.append(out["trace"][0])
        with contextlib.redirect_stdout(buf):
            est.partial_fit(X[a:b], y[a:b], classes=[-1.0, 1.0])
        PF._assert_close(est, P, w, it)
    got = parse_traces(buf.getvalue())
    assert len(got) == 1
    planned = reg in ("l1", "squaredl12")
    check_loss_trace(f"partial_fit_{reg}", f"partial_fit, {'planned' if planned else 'dense'} path, chunks {sizes}",
                     got[0], want, "planned" if planned else "dense")


def _sharded_worker(rank, world, port, out_dir, n_dev):
    import sys
    import torch
    import torch.distributed as dist
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank % n_dev)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    import sparsepoly_b200 as S
    from sparsepoly_b200 import distributed, synth
    distributed.enable_sharding()
    res = {}
    for tag, kw in _SHARDED:
        X = synth.criteo_like(_SH_N, _SH_D, 21 + rank)
        y = np.where(np.random.RandomState(31 + rank).rand(_SH_N) < 0.3, 1.0, -1.0)
        buf = io.StringIO()
        with warnings.catch_warnings(), contextlib.redirect_stdout(buf):
            warnings.simplefilter("ignore")
            S.SparseFactorizationMachineClassifier(random_state=rank, verbose=True, **kw).fit(X, y)
        res[tag] = np.array(parse_traces(buf.getvalue())[0])
    np.savez(os.path.join(out_dir, f"rank{rank}.npz"), **res)
    dist.barrier()
    dist.destroy_process_group()


_SH_N, _SH_D = 3000, 1200
_SHARDED = [
    ("sql12", dict(degree=2, loss="logistic", n_components=8, solver="psgd", regularizer="squaredl12", alpha=1e-4,
                   beta=1e-4, gamma=1e-3, eta0=0.1, max_iter=3, tol=-1.0, n_iter_no_change=10 ** 9, batch_size=512)),
    ("l1_deg3", dict(degree=3, loss="logistic", n_components=4, solver="psgd", regularizer="l1", alpha=1e-4,
                     beta=1e-4, gamma=1e-4, eta0=0.1, max_iter=3, tol=-1.0, n_iter_no_change=10 ** 9, batch_size=1000,
                     fit_lower="explicit")),
]


def test_sharded_psgd_epoch_losses_match_oracle(tmp_path):
    """Two ranks: each epoch's loss is summed over the ranks and divided by the global sample count; against the
    oracle on the interleaved data set."""
    import torch
    import torch.multiprocessing as mp
    from oracle import oracle as O
    from sparsepoly_b200 import synth
    from sparsepoly_b200.distributed import interleave_shards
    world = 2
    if torch.cuda.device_count() < world:
        pytest.skip("needs one GPU per rank")
    port = 35500 + (os.getpid() % 2000)
    mp.spawn(_sharded_worker, args=(world, port, str(tmp_path), torch.cuda.device_count()), nprocs=world, join=True)
    z = [np.load(tmp_path / f"rank{r}.npz") for r in range(world)]
    Xs = [synth.criteo_like(_SH_N, _SH_D, 21 + r) for r in range(world)]
    ys = [np.where(np.random.RandomState(31 + r).rand(_SH_N) < 0.3, 1.0, -1.0) for r in range(world)]
    for tag, kw in _SHARDED:
        b_loc = kw["batch_size"] // world
        order = interleave_shards([np.arange(_SH_N) + r * _SH_N for r in range(world)], b_loc * world)
        Xall, yall = sp.vstack(Xs).tocsr()[order], np.concatenate(ys)[order]
        out = O.fit_fm(Xall, yall, random_state=0, **dict(kw, batch_size=b_loc * world))
        for r in range(world):
            check_loss_trace(f"sharded_{tag}_rank{r}", "sharded psgd planned path, 2 ranks", list(z[r][tag]),
                             out["trace"], "planned")


# ============================================================================ 6. fits that stop on the trace
def _check_stop(tag, path, est, X, y, got, warned, out, want_stop, rule):
    """A fit with the chosen parameters against the oracle's fit with them and the replay of its trace."""
    assert out["n_iter_"] == want_stop and out["converged"] == (rule != "never")
    assert est.n_iter_ == out["n_iter_"] == len(got) - 1, (tag, est.n_iter_, out["n_iter_"], got)
    assert warned == (not out["converged"]), (tag, warned, out["converged"])
    if "it_" in out:
        assert est.it_ == out["it_"]
    assert rel_err(est.P_, out["P_"]) <= TOL and same_support(est.P_, out["P_"])
    if "w_" in out and hasattr(est, "w_"):
        assert rel_err(est.w_, out["w_"]) <= TOL
    _check_objective(est, X, y, out["P_"], out.get("w_"))
    print(f"{tag} [{path}] {rule}: device stops after epoch {est.n_iter_}, oracle after {out['n_iter_']}, "
          f"converged {out['converged']}")


def _viol_choice(trace, rule):
    """(tol, stop epoch, margin) of the named choice over a tol=-1 trace."""
    if rule == "never":
        tol, margin = tol_never(trace)
        return tol, len(trace) - 1, margin
    e = 0 if rule == "epoch0" else first_drop(trace)
    tol, margin = tol_stopping_at(trace, e)
    return tol, e, margin


E_STOP = 8
VIOL_STOP = [
    # (tag, path, oracle + estimator factory, env)
    ("pcd_cluster_fm3", "pcd cluster sweep", ("fm", PCD_CLF_PROB, dict(_FM3, max_iter=E_STOP)),
     dict(SPARSEPOLY_B200_SWEEP="cluster")),
    ("pcd_window_sql12", "pcd window sweep, speculative",
     ("fm", dict(WINDOW_PROB, degree=2, clf=False), dict(SPEC_CASES[1][3], max_iter=6)),
     dict(SPARSEPOLY_B200_SWEEP="window")),
    ("pbcd_cluster_k33_l21", "pbcd cluster sweep KCH=2", ("fm", PBCD_PROB, _pbcd_kw(33, 3, "l21", max_iter=E_STOP)),
     dict(SPARSEPOLY_B200_SWEEP="cluster")),
    ("pbcd_window_k8_omegacs", "pbcd window sweep",
     ("fm", PBCD_WINDOW_PROB, _pbcd_kw(8, 2, "omegacs", gamma=1e-6, max_iter=6)), dict(SPARSEPOLY_B200_SWEEP="window")),
    ("all_pcd_clf", "all-subsets pcd", ("all", dict(ALL_PROB, clf=True),
                                        dict(ALL_CASES[1][2], mean=True, max_iter=E_STOP, tol=-1.0, random_state=0)),
     {}),
    ("all_pbcd_reg", "all-subsets pbcd", ("all", dict(ALL_PROB, clf=False),
                                          dict(ALL_CASES[2][2], loss="squared", mean=True, max_iter=E_STOP, tol=-1.0,
                                               random_state=0)), {}),
]


def _viol_case(spec):
    kind, prob, kw = spec
    if kind == "fm":
        X, y, ref = _fm_oracle(prob, kw)
        return X, y, ref, kw, lambda k: (_pbcd_estimator(k, k["degree"]) if k["solver"] == "pbcd"
                                         else _fm_estimator(k))
    kw = dict(kw, loss=kw.get("loss", "squared"))
    X, y, ref = _all_oracle(prob, kw)
    return X, y, ref, kw, _all_estimator


@pytest.mark.parametrize("rule", ["epoch0", "first_drop", "never"])
@pytest.mark.parametrize("tag,path,spec,env", VIOL_STOP, ids=[c[0] for c in VIOL_STOP])
def test_fit_stops_on_violation_like_oracle(tag, path, spec, env, rule, monkeypatch):
    from oracle import oracle as O
    _with_env(monkeypatch, env)
    X, y, ref, kw, make = _viol_case(spec)
    tol, stop, margin = _viol_choice(ref["trace"], rule)
    assert replay_viol(ref["trace"], tol) == (stop, rule != "never")
    okw = dict(kw, tol=tol)
    okw.setdefault("loss", "squared")
    out = (O.fit_fm if spec[0] == "fm" else O.fit_all_subsets)(X, y, **okw)
    est = make(dict(kw, tol=tol))
    got, warned, _ = trace_of(est, X, y)
    print(f"{tag}: tol {tol!r} (smallest decision margin {margin:.3g}), replay stops after epoch {stop}")
    _check_stop(tag, path, est, X, y, got, warned, out, stop, rule)


PLATEAU_STOP = [
    # aggressive constant steps with shuffling: the planned case's epoch loss rises, and in both the chosen tol
    # lets the no-improvement count run up and reset before it stops the fit (eta0=2 diverges on the l21 case)
    ("psgd_planned_l1", "psgd planned path", _psgd_kw("l1", 8, eta0=2.0, learning_rate="constant", shuffle=True,
                                                      max_iter=10, batch_size=500)),
    ("psgd_dense_l21", "psgd dense-gradient path", _psgd_kw("l21", 16, eta0=1.0, learning_rate="constant",
                                                            shuffle=True, max_iter=10, batch_size=500)),
]


@pytest.mark.parametrize("n_iter_no_change", [1, 2, 3])
@pytest.mark.parametrize("tag,path,kw", PLATEAU_STOP, ids=[c[0] for c in PLATEAU_STOP])
def test_psgd_fit_stops_on_plateau_like_oracle(tag, path, kw, n_iter_no_change):
    from oracle import oracle as O
    X, y, ref = _psgd_oracle(kw)
    tol, stop, margin, resets = choose_plateau_tol(ref["trace"], n_iter_no_change)
    okw = dict(kw, tol=tol, n_iter_no_change=n_iter_no_change)
    out = O.fit_fm(X, y, **okw)
    assert replay_plateau(ref["trace"], tol, n_iter_no_change) == (stop, True, resets)
    est = _fm_estimator(okw)
    got, warned, _ = trace_of(est, X, y)
    assert ("plan_bytes" in est._psgd_stats) == (kw["regularizer"] == "l1")
    print(f"{tag}: n_iter_no_change {n_iter_no_change}, tol {tol!r} (smallest decision margin {margin:.3g}, "
          f"{resets} resets), replay stops after epoch {stop}")
    _check_stop(tag, path, est, X, y, got, warned, out, stop, "plateau")


def test_psgd_plateau_choices_reset_the_count():
    """In every PLATEAU_STOP case some chosen tol resets the no-improvement count; the planned case's loss rises."""
    rises = {}
    for tag, _, kw in PLATEAU_STOP:
        _, _, ref = _psgd_oracle(kw)
        rises[tag] = any(b > a for a, b in zip(ref["trace"], ref["trace"][1:]))
        assert any(choose_plateau_tol(ref["trace"], n)[3] > 0 for n in (2, 3)), tag
    assert rises["psgd_planned_l1"], rises


@pytest.mark.parametrize("solver", ["pcd", "pbcd"])
def test_fit_many_models_stop_on_their_own_violation(solver):
    """One fit_many call whose models stop after epochs 0, 1, 3 and never, each against its own oracle fit."""
    import sparsepoly_b200 as S
    from oracle import oracle as O
    E = 6
    reg = "omegati" if solver == "pcd" else "l21"
    kw = dict(degree=2, n_components=4, solver=solver, regularizer=reg, alpha=1e-3, beta=1e-4, gamma=1e-5,
              max_iter=E, random_state=0, mean=True)
    prob = dict(n=20000, d=2000, r=10, seed=11, kernel="anova", degree=2, clf=False)
    X, y, ref = _fm_oracle(prob, dict(kw, tol=-1.0))
    trace = ref["trace"]
    stops = [0, 1, 3, None]
    tols = [tol_stopping_at(trace, e)[0] if e is not None else tol_never(trace)[0] for e in stops]
    ests = [S.SparseFactorizationMachineRegressor(tol=t, verbose=True, **kw) for t in tols]
    buf = io.StringIO()
    with warnings.catch_warnings(record=True) as caught, contextlib.redirect_stdout(buf):
        warnings.simplefilter("always")
        S.fit_many(ests, X, y)
    traces = parse_traces(buf.getvalue())
    assert len(traces) == len(ests) and _not_converged(caught) == 1
    for e, tol, est, got in zip(stops, tols, ests, traces):
        out = O.fit_fm(X, y, loss="squared", tol=tol, **kw)
        stop = E - 1 if e is None else e
        assert est.n_iter_ == out["n_iter_"] == stop == len(got) - 1, (e, est.n_iter_, out["n_iter_"])
        assert out["converged"] == (e is not None)
        assert rel_err(est.P_, out["P_"]) <= TOL and same_support(est.P_, out["P_"])
        assert rel_err(est.w_, out["w_"]) <= TOL
        check_viol_trace(f"fit_many_{solver}_stop{e}", f"fit_many {solver}, tol {tol!r}", got, out, est)
        _check_objective(est, X, y, out["P_"], out["w_"])
