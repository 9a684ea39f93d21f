"""Every compiled variant of the hot-path templates against the C oracle, and the row kernels against the exact
reference of tests/test_exact_reference_cpu.py.

Each template instantiation is separate code (register arrays, unroll counts, shuffle masks, shared-memory
sizes), so each one needs a run of its own:
  * rows.cu rows_all_kernel<DEG, G, MODE> (predict, Gram matrix): G = 8 / 16 / 32 and the loop over component chunks
    for k > 32 (rows_pbcd_cache_kernel<DEG, G> runs the same body through the pbcd fits below)
  * pcd.cu launch_sweep<KIND, 5, LOSS, NZ> (NZ = 1 and 2) and pcd_window.cu at degree 5
  * pbcd.cu launch_block<KIND, DEG, KCH> with KCH = 2 / 4 (k in 33..128), degree 5; pbcd_window.cu at degree 5
  * psgd.cu psgd_grad_kernel<DEG, NORD, G, KCH>: G = 16 / 32, KCH = 1 / 2 / 4, NORD = 1..4 (the only path of
    l21 / squaredl21)
  * psgd_plan.cu launch_minibatch at degree 5, squaredl12 at k = 63..128
Every test asserts that it reached the variant it names (plan mode, geometry, the NZ choice of pick_nz,
kernel-class launch counts of sp_profile_*), so that a silent fall-back to another path fails."""
import ctypes as C
import math

import numpy as np
import pytest
import scipy.sparse as sp

from golden_util import rel_err, same_support
from test_exact_reference_cpu import (ROW_NNZ, assert_within, dp_bound, exact_kernel, exact_linear,
                                      exact_prediction, prediction_bound, rows_matrix, signed_P)
from test_parity_gpu import _check_objective, _fit, _problem, _wspec_read

pytestmark = pytest.mark.gpu

TOL = 1e-9
ROW_KS = [1, 7, 8, 9, 16, 17, 32, 33, 64, 100, 128]
DEGREES = [1, 2, 3, 4, 5, -1]

# kernel classes of sp_profile_* (csrc/common.cuh)
PROF_SWEEP_PBCD, PROF_PSGD_GRAD = 3, 4


def _profile(on):
    from sparsepoly_b200 import _lib
    _lib.check(_lib.load().sp_profile_enable(int(on)))


def _launches():
    from sparsepoly_b200 import _lib
    ms, cnt = (C.c_double * 8)(), (C.c_longlong * 8)()
    _lib.check(_lib.load().sp_profile_collect(ms, cnt))
    return list(cnt)


def _fit_profiled(est, X, y):
    _profile(True)
    try:
        _fit(est, X, y)
        cnt = _launches()
    finally:
        _profile(False)
    return est, cnt


_ORACLE = {}


def _oracle(key, fn):
    """Oracle fits are shared by every geometry of the same problem (the host oracle is the cost)."""
    if key not in _ORACLE:
        _ORACLE[key] = fn()
    return _ORACLE[key]


def _fm_estimator(kw):
    import sparsepoly_b200 as S
    clf = kw.get("loss", "squared") != "squared"
    ekw = dict(kw)
    if not clf:
        ekw.pop("loss", None)
    return (S.SparseFactorizationMachineClassifier if clf else S.SparseFactorizationMachineRegressor)(**ekw)


def _compare(est, out, X, y, check_objective=True):
    """P_, w_, support and the iteration counters of a CUDA fit against the oracle's; returns (err, frac)."""
    err = rel_err(est.P_, out["P_"])
    assert err <= TOL, err
    assert same_support(est.P_, out["P_"])
    if "w_" in out and hasattr(est, "w_"):
        assert rel_err(est.w_, out["w_"]) <= TOL
    assert est.n_iter_ == out["n_iter_"]
    if "it_" in out:
        assert est.it_ == out["it_"]
    if check_objective:
        _check_objective(est, X, y, out["P_"], out.get("w_"))
    return err, float(np.mean(out["P_"] != 0))


def _pick_nz(ds, n_cta, threads):
    """Python restatement of pick_nz (csrc/pcd.cu)."""
    avg = ds.nnz / max(ds.n_features, 1)
    return 2 if avg / n_cta > 0.8 * threads else 1


# ============================================================================ a. row DP kernels (rows.cu)
def _dp_numpy(X, P_dk, degree):
    """rows_all_body.inc for PX=false, transliterated: A[t] += (A[t-1] * x) * p over the row's features in
    ascending order (t descending), all-subsets A *= 1 + x * p.  Separate IEEE fp64 operations, as the
    library is built with -fmad=false."""
    X = sp.csr_matrix(X)
    n, k = X.shape[0], P_dk.shape[1]
    m = degree if degree > 0 else 1
    out = np.empty((n, k))
    for i in range(n):
        A = np.zeros((m + 1, k))
        A[0] = 1.0
        if degree == -1:
            A[1] = 1.0
        for e in range(X.indptr[i], X.indptr[i + 1]):
            x, p = X.data[e], P_dk[X.indices[e]]
            if degree == -1:
                A[1] = A[1] * (1.0 + x * p)
            else:
                for t in range(m, 0, -1):
                    A[t] = A[t] + (A[t - 1] * x) * p
        out[i] = A[m]
    return out


@pytest.mark.parametrize("k", ROW_KS)
def test_kernel_matrix_bitwise_and_within_exact_bound(k):
    """sp_kernel_matrix (MODE 2): bit-identical to the NumPy transliteration of the recurrence, and within
    the rounding bound of the exact value, on rows of 0..200 nonzeros and one with |x p| ~ 1e3."""
    from sparsepoly_b200 import kernels
    X = rows_matrix(seed=k)
    assert sorted(set(np.diff(X.indptr))) == sorted(set(ROW_NNZ) | {9})
    for degree in DEGREES:
        P = signed_P(X.shape[1], k, 100 + k, degree)
        got = kernels.all_subsets_kernel(X, P.T) if degree == -1 else kernels.anova_kernel(X, P.T, degree)
        assert got.shape == (X.shape[0], k)
        want_bits = _dp_numpy(X, P, degree)
        bad = np.argwhere(got != want_bits)
        assert bad.size == 0, (degree, bad[:5].tolist(), got[tuple(bad[0])], want_bits[tuple(bad[0])])
        exact, abs_ref = exact_kernel(X, P, degree)
        assert_within(got, exact, dp_bound(X, abs_ref, degree), f"kernel k={k} degree={degree}")


@pytest.mark.parametrize("k", ROW_KS)
def test_predict_within_exact_bound(k):
    """sp_predict (MODE 0; components summed with a shuffle tree): kernels.poly_predict and
    solvers.poly_predict without / with w, out_stride=3, accumulate=True onto a nonzero out."""
    import torch
    from sparsepoly_b200 import kernels, solvers
    from sparsepoly_b200.dataset import DeviceDataset
    X = rows_matrix(seed=200 + k)
    n, d = X.shape
    rng = np.random.RandomState(k)
    lams = np.where(rng.rand(k) < 0.5, -1.0, 1.0)
    w = rng.randn(d)
    lin, lin_abs = exact_linear(X, w)
    ds = DeviceDataset(X, need_csr=True, need_csc=False)
    lams_dev = torch.from_numpy(lams).cuda()
    w_dev = torch.from_numpy(w).cuda()
    for degree in DEGREES:
        P = signed_P(d, k, 300 + k, degree)
        exact, abs_ref = exact_kernel(X, P, degree)
        want = exact_prediction(exact, lams)
        bound = prediction_bound(X, abs_ref, lams, degree)
        kern = ("all-subsets", 2) if degree == -1 else ("anova", degree)
        assert_within(kernels.poly_predict(X, P.T, lams, *kern), want, bound, f"kernels.poly_predict {degree}")
        P_dev = torch.from_numpy(np.ascontiguousarray(P)).cuda()
        got = solvers.poly_predict(ds, P_dev, lams_dev, degree).cpu().numpy()
        assert_within(got, want, bound, f"solvers.poly_predict w=None degree {degree}")
        want_w = exact_prediction(exact, lams, lin)
        bound_w = prediction_bound(X, abs_ref, lams, degree, linear_abs=lin_abs)
        got = solvers.poly_predict(ds, P_dev, lams_dev, degree, w=w_dev).cpu().numpy()
        assert_within(got, want_w, bound_w, f"solvers.poly_predict with w, degree {degree}")
        # strided output: only slots 0, 3, 6, ... are written
        base = rng.randn(3 * n)
        out = torch.from_numpy(base.copy()).cuda()
        solvers.poly_predict(ds, P_dev, lams_dev, degree, w=w_dev, out=out, out_stride=3)
        o = out.cpu().numpy()
        assert_within(o[0::3], want_w, bound_w, f"out_stride=3 degree {degree}")
        assert np.array_equal(o[1::3], base[1::3]) and np.array_equal(o[2::3], base[2::3])
        # accumulate onto a nonzero out: out + pred, untouched slots untouched
        first = o[0::3].copy()
        solvers.poly_predict(ds, P_dev, lams_dev, degree, w=w_dev, out=out, out_stride=3, accumulate=True)
        o2 = out.cpu().numpy()
        assert np.array_equal(o2[0::3], first + first)
        assert np.array_equal(o2[1::3], base[1::3]) and np.array_equal(o2[2::3], base[2::3])
        out1 = torch.from_numpy(base[0::3].copy()).cuda()
        solvers.poly_predict(ds, P_dev, lams_dev, degree, out=out1, accumulate=True)
        pred = solvers.poly_predict(ds, P_dev, lams_dev, degree).cpu().numpy()
        assert np.array_equal(out1.cpu().numpy(), base[0::3] + pred)


# ============================================================================ b. pcd at degree 5
# (beta, gamma) per regularizer.  The fits use explicit lower orders.  Without them only the degree-5 weights
# exist; starting at 0.01 their gradients are ~1e-8, so beta and gamma must be tiny for the model to leave zero,
# and the Newton steps then divide by curvatures of ~1e-16: on this problem the oracle itself turns a 1-ulp
# change of the starting point into a change of 1e3..1e12 ulps of P_ within two epochs (fit_lower="augment" or
# None), so a 1e-9 comparison would test the conditioning, not the kernels.
PCD5_REG = {"l1": (1e-4, 1e-5), "omegati": (1e-4, 1e-6)}
PCD5_CASES = [(loss, reg, "explicit") for loss in ("squared", "logistic", "squared_hinge")
              for reg in ("l1", "omegati")]


def _pcd5_kw(loss, reg, fit_lower, **extra):
    beta, gamma = PCD5_REG[reg]
    kw = dict(degree=5, loss=loss, n_components=4, solver="pcd", regularizer=reg, alpha=1e-4, beta=beta,
              gamma=gamma, max_iter=2, tol=-1.0, random_state=0, mean=True, fit_lower=fit_lower)
    kw.update(extra)
    return kw


def _fm_case(prob, kw):
    """(X, y, oracle output) of a seeded problem; the oracle fit is cached."""
    from oracle import oracle as O
    X, y = _problem(**prob)
    okw = dict(kw)
    okw.setdefault("loss", "squared")
    out = _oracle(repr((sorted(prob.items()), sorted(okw.items(), key=str))), lambda: O.fit_fm(X, y, **okw))
    return X, y, out


PCD5_PROB = dict(n=20000, d=2000, r=10, seed=7, kernel="anova", degree=3)


@pytest.mark.parametrize("nz,n_cta,threads", [(1, 1, 256), (2, 1, 32), (2, 2, 32), (1, 4, 64)])
@pytest.mark.parametrize("loss,reg,fit_lower", PCD5_CASES)
def test_pcd_degree5_cluster_sweep(loss, reg, fit_lower, nz, n_cta, threads, monkeypatch):
    """launch_sweep<KIND_FM, 5, LOSS, NZ> (and the lower orders 2..4) for the three losses and l1 / omegati;
    NZ = 2 is taken once the mean column slice exceeds 0.8 * threads (pick_nz)."""
    monkeypatch.setenv("SPARSEPOLY_B200_SWEEP", "cluster")
    monkeypatch.setenv("SPARSEPOLY_B200_NCTA", str(n_cta))
    monkeypatch.setenv("SPARSEPOLY_B200_THREADS", str(threads))
    kw = _pcd5_kw(loss, reg, fit_lower)
    X, y, out = _fm_case(dict(PCD5_PROB, clf=loss != "squared"), kw)
    est = _fit(_fm_estimator(kw), X, y)
    plan, ds = est._dev_state["plan"], est._dev_state["ds"]
    assert plan.mode == "cluster" and (plan.n_cta, plan.threads) == (n_cta, threads)
    assert _pick_nz(ds, plan.n_cta, plan.threads) == nz
    err, frac = _compare(est, out, X, y)
    assert 0.01 < frac < 0.99, frac
    print(loss, reg, fit_lower, "NZ", nz, "err", err, "nonzero fraction", frac)


PCD5_WINDOW_PROB = dict(n=100000, d=5000, r=10, seed=5, kernel="anova", degree=3)
PCD5_WINDOW_CASES = [("squared", "omegati", "explicit"), ("logistic", "l1", "explicit"),
                     ("squared_hinge", "omegati", "explicit")]


@pytest.mark.parametrize("horizon,near", [(0, 0), (0, 1), (0, 2), (1, 0), (1, 1), (1, 2)])
@pytest.mark.parametrize("loss,reg,fit_lower", PCD5_WINDOW_CASES)
def test_pcd_degree5_window_sweep(loss, reg, fit_lower, horizon, near, monkeypatch):
    """wdispatch_loss at degree 5 (pcd_window.cu): the cached orders A^1..A^4 fill the whole record."""
    monkeypatch.setenv("SPARSEPOLY_B200_SWEEP", "window")
    monkeypatch.setenv("SPARSEPOLY_B200_HORIZON", str(horizon))
    monkeypatch.setenv("SPARSEPOLY_B200_NEAR", str(near))
    kw = _pcd5_kw(loss, reg, fit_lower, gamma=PCD5_REG[reg][1] / 10)
    X, y, out = _fm_case(dict(PCD5_WINDOW_PROB, clf=loss != "squared"), kw)
    est = _fit(_fm_estimator(kw), X, y)
    plan = est._dev_state["plan"]
    assert plan.mode == "window", plan.wplan.stats
    assert plan.wplan.stats["horizon"] == horizon and plan.wplan.stats["near"] == near, plan.wplan.stats
    err, frac = _compare(est, out, X, y)
    assert 0.01 < frac < 0.99, frac
    print(loss, reg, fit_lower, plan.wplan.stats, "err", err, "nonzero fraction", frac)


def test_pcd_degree5_zero_update_speculation(monkeypatch):
    """Degree 5 in a regime where most coordinates sit at zero after the first epoch: the window engine
    speculates on zero updates and ends with the model of the non-speculative sweep."""
    monkeypatch.setenv("SPARSEPOLY_B200_SWEEP", "window")
    kw = dict(degree=5, n_components=4, solver="pcd", regularizer="omegati", alpha=1e-4, beta=1e-4, gamma=1e-6,
              max_iter=4, tol=-1.0, random_state=0, mean=True, fit_lower="explicit")
    X, y, out = _fm_case(dict(PCD5_WINDOW_PROB, clf=False), kw)
    _wspec_read()
    est = _fit(_fm_estimator(kw), X, y)
    n_spec, n_rej = _wspec_read()
    assert est._dev_state["plan"].mode == "window"
    err, frac = _compare(est, out, X, y)
    assert 0.0 < frac < 0.2, frac
    assert n_spec > 0, "speculation never engaged"
    assert n_rej < n_spec
    monkeypatch.setenv("SPARSEPOLY_B200_SPEC", "0")
    est0 = _fit(_fm_estimator(kw), X, y)
    assert _wspec_read() == (0, 0)
    assert rel_err(est.P_, est0.P_) <= 1e-11 and rel_err(est.w_, est0.w_) <= 1e-11
    assert np.array_equal(est.P_ != 0, est0.P_ != 0)
    print("nonzero fraction", frac, "speculated positions", n_spec, "rejected", n_rej, "err", err)


# ============================================================================ c. pbcd: k > 32 and degree 5
PBCD_GAMMA = {"l1": 1e-5, "l21": 1e-4, "omegacs": 1e-6, "squaredl21": 1e-6}
# all-subsets: the l1 / l21 block prox needs a much larger gamma to zero rows, l21 growing with k
PBCD_ALL_GAMMA = {"l1": lambda k: 3e-2, "l21": lambda k: {33: 0.3, 64: 1.0, 65: 1.0, 100: 2.0, 128: 3.0}[k],
                  "omegacs": lambda k: 1e-6}
PBCD_PROB = dict(n=5000, d=1000, r=10, seed=9, kernel="anova", degree=3, clf=False)
PBCD_WIDE = ([(k, deg, reg) for k in (33, 64, 65, 100, 128) for deg in (2, 3, 5, -1)
              for reg in ("l1", "l21", "omegacs")] + [(k, 2, "squaredl21") for k in (33, 64, 65, 100, 128)])


def _pbcd_kw(k, degree, reg, **extra):
    gamma = PBCD_GAMMA[reg] if degree != -1 else PBCD_ALL_GAMMA[reg](k)
    kw = dict(n_components=k, solver="pbcd", regularizer=reg, beta=1e-4, gamma=gamma, max_iter=2,
              tol=-1.0, random_state=0, mean=True)
    if degree != -1:
        kw.update(degree=degree, alpha=1e-4)
    kw.update(extra)
    return kw


def _pbcd_case(prob, kw, degree):
    from oracle import oracle as O
    if degree != -1:
        return _fm_case(prob, kw)
    X, y = _problem(**dict(prob, kernel="all"))
    okw = dict(kw, loss="squared")
    out = _oracle(repr((sorted(prob.items()), sorted(okw.items(), key=str), "all")),
                  lambda: O.fit_all_subsets(X, y, **okw))
    return X, y, out


def _pbcd_estimator(kw, degree):
    import sparsepoly_b200 as S
    return _fm_estimator(kw) if degree != -1 else S.SparseAllSubsetsRegressor(**kw)


def _check_pbcd_launches(cnt, kw, degree):
    n_orders = degree - 1 if (degree != -1 and kw.get("fit_lower", "explicit") == "explicit") else 1
    assert cnt[PROF_SWEEP_PBCD] == kw["max_iter"] * n_orders, cnt


@pytest.mark.parametrize("k,degree,reg", PBCD_WIDE)
def test_pbcd_wide_cluster_sweep(k, degree, reg):
    """dispatch_kch with KCH = 2 (k <= 64) and KCH = 4 (k <= 128); SweepPlan forces the cluster sweep for
    k > 32."""
    kw = _pbcd_kw(k, degree, reg)
    X, y, out = _pbcd_case(PBCD_PROB, kw, degree)
    est, cnt = _fit_profiled(_pbcd_estimator(kw, degree), X, y)
    plan = est._dev_state["plan"]
    assert plan.mode == "cluster" and plan.wplan is None
    _check_pbcd_launches(cnt, kw, degree)
    err, frac = _compare(est, out, X, y)
    assert 0.01 < frac < 0.99, frac
    print(k, degree, reg, "KCH", -(-k // 32), "err", err, "nonzero fraction", frac)


@pytest.mark.parametrize("n_cta,threads", [(1, 32), (16, 32), (16, 256)])
def test_pbcd_k128_degree5_geometries(n_cta, threads, monkeypatch):
    """k = 128, degree 5 on the smallest and largest cluster geometries: (16, 256) has the largest dynamic
    shared memory of launch_block and the largest Av register block."""
    monkeypatch.setenv("SPARSEPOLY_B200_NCTA", str(n_cta))
    monkeypatch.setenv("SPARSEPOLY_B200_THREADS", str(threads))
    kw = _pbcd_kw(128, 5, "omegacs")
    X, y, out = _pbcd_case(PBCD_PROB, kw, 5)
    est, cnt = _fit_profiled(_pbcd_estimator(kw, 5), X, y)
    plan = est._dev_state["plan"]
    assert plan.mode == "cluster" and (plan.n_cta, plan.threads) == (n_cta, threads)
    _check_pbcd_launches(cnt, kw, 5)
    err, frac = _compare(est, out, X, y)
    assert 0.01 < frac < 0.99, frac


PBCD_WINDOW_PROB = dict(n=50000, d=5000, r=8, seed=6, kernel="anova", degree=3, clf=False)


@pytest.mark.parametrize("horizon", [0, 1])
@pytest.mark.parametrize("k,reg", [(5, "omegacs"), (32, "l21"), (32, "omegacs")])
def test_pbcd_degree5_window_sweep(k, reg, horizon, monkeypatch):
    """launch_bw<5> (pbcd_window.cu) for k = 5 and 32, explicit lower orders."""
    monkeypatch.setenv("SPARSEPOLY_B200_SWEEP", "window")
    monkeypatch.setenv("SPARSEPOLY_B200_HORIZON", str(horizon))
    kw = _pbcd_kw(k, 5, reg, gamma=PBCD_GAMMA[reg] / 10)
    X, y, out = _pbcd_case(PBCD_WINDOW_PROB, kw, 5)
    est, cnt = _fit_profiled(_pbcd_estimator(kw, 5), X, y)
    plan = est._dev_state["plan"]
    assert plan.mode == "window" and plan.wplan.stats["horizon"] == horizon, plan.wplan.stats
    _check_pbcd_launches(cnt, kw, 5)
    err, frac = _compare(est, out, X, y)
    assert 0.01 < frac < 0.99, frac
    print(k, reg, plan.wplan.stats, "err", err, "nonzero fraction", frac)


# ============================================================================ d. psgd, dense-gradient path
PSGD_N, PSGD_D, PSGD_BATCH = 20000, 4000, 2000
PSGD_GAMMA = {"l21": 1e-3, "squaredl21": 3e-4, "l1": 2e-4, "squaredl12": 1e-3}
PSGD_DENSE = ([("l21", k, 2, "explicit") for k in (16, 17, 32, 33, 64, 128)]
              + [("squaredl21", k, 2, "explicit") for k in (16, 17, 32, 33, 64, 128)]
              + [("l21", 17, 3, "explicit"), ("l21", 64, 4, "explicit"), ("l21", 128, 5, "explicit"),
                 ("l21", 33, 5, None)]
              + [("l1", 128, 2, "explicit"), ("squaredl12", 128, 2, "explicit")])
DENSE_ERRORS = {}


def _psgd_case(reg, k, degree, fit_lower, seed=1, **extra):
    from oracle import oracle as O
    from sparsepoly_b200 import synth
    X = synth.criteo_like(PSGD_N, PSGD_D, seed)
    y = np.where(np.random.RandomState(seed + 1).rand(PSGD_N) < 0.3, 1.0, -1.0)
    kw = dict(degree=degree, loss="logistic", n_components=k, solver="psgd", regularizer=reg, alpha=1e-4,
              beta=1e-4, gamma=PSGD_GAMMA[reg], eta0=0.1, max_iter=2, tol=-1.0, random_state=0,
              n_iter_no_change=10 ** 9, batch_size=PSGD_BATCH, fit_lower=fit_lower)
    kw.update(extra)
    out = _oracle(repr(("psgd", seed, sorted(kw.items(), key=str))), lambda: O.fit_fm(X, y, **kw))
    return X, y, kw, out


@pytest.mark.parametrize("reg,k,degree,fit_lower", PSGD_DENSE)
def test_psgd_dense_gradient_path(reg, k, degree, fit_lower, monkeypatch):
    """psgd_grad_kernel<DEG, NORD, G, KCH>: G = 16 for k <= 16, else 32; KCH = ceil(k / 32); NORD = degree - 1
    with explicit lower orders.  Gradients are summed with fp64 atomics in no fixed order."""
    from sparsepoly_b200 import solvers
    from sparsepoly_b200.dataset import DeviceDataset
    if reg in solvers.PLANNED_REGS:
        monkeypatch.setattr(solvers, "PLANNED_REGS", ())
    X, y, kw, out = _psgd_case(reg, k, degree, fit_lower)
    est, cnt = _fit_profiled(_fm_estimator(kw), X, y)
    assert "plan_bytes" not in est._psgd_stats, est._psgd_stats            # not the planned path
    n_mb = math.ceil(PSGD_N / PSGD_BATCH)
    assert cnt[PROF_PSGD_GRAD] == kw["max_iter"] * n_mb, cnt
    nord = degree - 1 if fit_lower == "explicit" else 1
    G, KCH = (16 if k <= 16 else 32), -(-k // 32)
    if KCH * nord == 1:           # the hot-feature pre-reduction runs: the 13 dense columns (and Zipf heads) are marked
        assert DeviceDataset(X, need_csr=True, need_csc=False).struct.n_hot_feat >= 13
    err = rel_err(est.P_, out["P_"])
    DENSE_ERRORS[(reg, k, degree, fit_lower)] = err
    print(f"dense psgd {reg} k={k} degree={degree} fit_lower={fit_lower} G={G} KCH={KCH} NORD={nord}: "
          f"max relative error of P_ {err:.3e}, w_ {rel_err(est.w_, out['w_']):.3e}")
    err, frac = _compare(est, out, X, y, check_objective=False)
    if reg != "l21":      # (the reference's l21 prox leaves rows at or below the threshold unchanged: never sparse)
        assert 0.01 < frac < 0.99, frac


# ============================================================================ e. psgd, planned path
PSGD_PLANNED = ([("squaredl12", k, 2, "explicit") for k in (63, 64, 65, 127, 128)]
                + [("l1", 128, 2, "explicit"), ("l1", 8, 5, "explicit"), ("l1", 40, 5, None),
                   ("squaredl12", 8, 5, None)])


@pytest.mark.parametrize("reg,k,degree,fit_lower", PSGD_PLANNED)
def test_psgd_planned_path_wide_and_degree5(reg, k, degree, fit_lower):
    """launch_minibatch at degree 5 (NORD 4 and 1), squaredl12 at k = 63..128 (odd k: the VEC=1 statistics
    pass; k = 128 fills s_bn[128]); fixed summation order, so two fits are bit-identical."""
    X, y, kw, out = _psgd_case(reg, k, degree, fit_lower, seed=3)
    est = _fit(_fm_estimator(kw), X, y)
    assert "plan_bytes" in est._psgd_stats, est._psgd_stats                # the planned path
    err, frac = _compare(est, out, X, y, check_objective=False)
    assert 0.01 < frac < 0.99, frac
    est2 = _fit(_fm_estimator(kw), X, y)
    assert np.array_equal(est.P_, est2.P_) and np.array_equal(est.w_, est2.w_)
    print(reg, k, degree, fit_lower, "err", err, "nonzero fraction", frac)


# ============================================================================ f. limits
@pytest.mark.parametrize("solver,reg,degree,k,match", [
    ("pcd", "omegati", 6, 4, "1..5"), ("pbcd", "omegacs", 6, 4, "1..5"), ("psgd", "l1", 6, 4, "2..5"),
    ("psgd", "l21", 6, 4, "2..5"), ("pbcd", "l21", 2, 129, "n_components=129 > 128"),
    ("psgd", "l21", 2, 129, "n_components=129 > 128"), ("psgd", "squaredl12", 2, 129, "n_components=129 > 128")])
def test_unsupported_degree_and_width_raise_and_process_recovers(solver, reg, degree, k, match):
    """degree > 5 and n_components > 128 fail with a ValueError naming the supported range; a valid fit in
    the same process still works afterwards."""
    from sparsepoly_b200 import synth
    X = synth.uniform_sparse(600, 80, 6, 2)
    y = np.random.RandomState(0).randn(600)
    kw = dict(degree=degree, n_components=k, solver=solver, regularizer=reg, alpha=1e-3, beta=1e-3, gamma=1e-3,
              max_iter=1, tol=-1.0, random_state=0)
    with pytest.raises(ValueError, match=match):
        _fit(_fm_estimator(kw), X, y)
    from oracle import oracle as O
    kw_ok = dict(kw, degree=3 if solver != "psgd" else 2, n_components=4)
    est = _fit(_fm_estimator(kw_ok), X, y)
    out = O.fit_fm(X, y, loss="squared", **kw_ok)
    assert rel_err(est.P_, out["P_"]) <= TOL and same_support(est.P_, out["P_"])
