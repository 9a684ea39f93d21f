"""The planned psgd path (csrc/psgd_plan.cu, host side psgd_plan.py) at its limits, against the C oracle:
  a. column classes at their boundaries (1, 2 / 8 / 9 nonzeros, one chunk of 63 / 64, 65 .. 129, a column of
     many chunks) for every (G, KCH) dispatch, and the minibatch edges: empty minibatches, a partial last one,
     batch_size=1, batch_size > n, shuffle=True, a plan built in several groups;
  b. every path of the squared-l1,2 selection: band hit, band miss (generic passes, the half-width doubles),
     band overflow (more than SP_PSGD_BAND_CAP values in one column's band: the half-width halves), odd / even
     k, several orders, d below one statistics block and above STAT_PART_MAX blocks;
  c. long horizons of the lazy frame: beta = 0 (thresholds unbounded), the scales crossing 1e100 at an epoch end,
     inside an epoch and inside one partial_fit call (the frame is folded, never overflows).
Every test asserts that it reached the path it names -- plan class counts, selection counters, the scales'
trajectory -- and prints them."""
import numpy as np
import pytest
import scipy.sparse as sp

from golden_util import rel_err
from test_kernel_variants_gpu import _compare, _fm_estimator, _oracle
from test_parity_gpu import _fit

pytestmark = pytest.mark.gpu

LENS = (1, 2, 8, 9, 63, 64, 65, 128, 129)       # nonzeros per minibatch of the class features
B = 256                                          # rows per minibatch of the class problem; feature len(LENS) is dense
FLAG = 1 << 30                                   # lc_cnt: the column's only chunk


def _oracle_fit(name, X, y, kw, **init):
    """The oracle's fit of a named problem, cached per (problem, settings, warm start)."""
    import hashlib
    from oracle import oracle as O
    key = repr((name, sorted(kw.items(), key=str), sorted((k, hashlib.sha1(v.tobytes()).hexdigest())
                                                          for k, v in init.items())))
    return _oracle(key, lambda: O.fit_fm(X, y, **kw, **init))


def _kw(**extra):
    kw = dict(degree=2, loss="logistic", n_components=8, solver="psgd", regularizer="squaredl12", alpha=1e-3,
              beta=1e-3, gamma=1e-3, eta0=0.1, learning_rate="constant", max_iter=2, tol=-1.0, random_state=0,
              n_iter_no_change=10 ** 9, batch_size=B, fit_lower=None)
    kw.update(extra)
    return kw


def _labels(n, seed):
    return np.where(np.random.RandomState(seed).rand(n) < 0.4, 1.0, -1.0)


def _class_problem(n_mb=4, tail=100, empty=(), seed=0):
    """In every full minibatch of B rows feature f has exactly LENS[f] nonzeros and feature len(LENS) all B (four
    chunks); 48 more features take 3 nonzeros per row.  Minibatches in `empty` are rows without nonzeros; the last
    one has `tail` rows."""
    rng = np.random.RandomState(seed)
    n = n_mb * B + tail
    n_extra = 48
    d = len(LENS) + 1 + n_extra
    rows, cols = [], []
    for m in range(n_mb + (1 if tail else 0)):
        r0, nb = m * B, min(B, n - m * B)
        if m in empty:
            continue
        for f, L in enumerate(LENS):
            sel = rng.choice(nb, min(L, nb), replace=False)
            rows.append(r0 + sel); cols.append(np.full(sel.size, f))
        rows.append(r0 + np.arange(nb)); cols.append(np.full(nb, len(LENS)))
        for i in range(nb):
            sel = len(LENS) + 1 + rng.choice(n_extra, 3, replace=False)
            rows.append(np.full(3, r0 + i)); cols.append(sel)
    rows, cols = np.concatenate(rows), np.concatenate(cols)
    X = sp.csr_matrix((rng.uniform(0.2, 1.0, rows.size), (rows, cols)), shape=(n, d))
    X.sum_duplicates()
    X.sort_indices()
    return X, _labels(n, seed + 1)


def _capture_plans(monkeypatch, group_entries=None):
    """fit keeps its plans in a closure: record every plan _psgd_plan builds (optionally in small build groups)."""
    from sparsepoly_b200 import estimators
    from sparsepoly_b200.psgd_plan import PsgdPlan
    plans = []

    def plan(m, data):
        extra = {} if group_entries is None else dict(group_entries=group_entries)
        p = PsgdPlan(data["ds"].csr, data["idx"], data["ds"].n_features, m["b_loc"], world=m["world"],
                     rank=m["rank"], group=m["group"], **extra)
        plans.append(p)
        return p
    monkeypatch.setattr(estimators._BaseSparseFactorizationMachine, "_psgd_plan", staticmethod(plan))
    return plans


def _record_frames(monkeypatch):
    """(C, Cw) of the context after every psgd_planned_run call."""
    from sparsepoly_b200 import solvers
    frames = []
    run = solvers.psgd_planned_run

    def wrapped(ctx, *a, **k):
        it = run(ctx, *a, **k)
        frames.append((ctx.struct.C, ctx.struct.Cw))
        return it
    monkeypatch.setattr(solvers, "psgd_planned_run", wrapped)
    return frames


def _class_counts(plan, m):
    """(columns by length, singles, short, chunks, flagged single chunks, multi-chunk columns) of minibatch m."""
    u0, u1 = plan.mb_uptr[m], plan.mb_uptr[m + 1]
    lens = np.diff(plan.u_ptr.cpu().numpy()[u0:u1 + 1])
    cnt = plan.lc_cnt.cpu().numpy()[plan.mb_lcptr[m]:plan.mb_lcptr[m + 1]]
    return (lens, int(plan.mb_sgptr[m + 1] - plan.mb_sgptr[m]), int(plan.mb_shptr[m + 1] - plan.mb_shptr[m]),
            int(cnt.size), int(np.sum(cnt >= FLAG)), int(plan.mb_mlptr[m + 1] - plan.mb_mlptr[m]))


def _assert_classes(plan, full_mbs):
    """Every full minibatch holds every class: the LENS lengths, a column of four chunks, singles, short columns,
    flagged single chunks (9..64 nonzeros) and multi-chunk columns (65.. nonzeros)."""
    out = []
    for m in full_mbs:
        lens, n_sg, n_sh, n_lc, n_flag, n_ml = _class_counts(plan, m)
        assert set(LENS) | {B} <= set(lens.tolist()), (m, sorted(set(lens.tolist())))
        assert n_sg >= 1 and n_sh >= 1 and n_flag >= 3 and n_ml >= 4, (m, n_sg, n_sh, n_flag, n_ml)
        assert n_lc == n_flag + int(np.sum(-(-lens[lens > 64] // 64)))
        out.append((n_sg, n_sh, n_lc, n_flag, n_ml))
    return out


def _fit_twice(kw, X, y, **init):
    """A CUDA fit and a second one bit-identical to it (fixed summation order)."""
    est = _fit_init(_fm_estimator(kw), X, y, **init)
    est2 = _fit_init(_fm_estimator(kw), X, y, **init)
    assert np.array_equal(est.P_, est2.P_) and np.array_equal(est.w_, est2.w_)
    return est


def _fit_init(est, X, y, P_init=None, w_init=None):
    if P_init is not None:
        est.warm_start = True
        est.P_ = P_init.copy()
        est.w_ = np.zeros(P_init.shape[2]) if w_init is None else w_init.copy()
    return _fit(est, X, y)


def _nonzero_fraction(est):
    frac = float(np.mean(est.P_ != 0))
    assert 0.0 < frac < 1.0, frac
    return frac


# ============================================================================ a. column classes, minibatch edges
CLASS_CASES = [(reg, degree, fit_lower, k) for reg in ("l1", "squaredl12")
               for degree, fit_lower in ((2, None), (4, "explicit"), (4, None)) for k in (8, 16, 32, 33, 128)]


@pytest.mark.parametrize("reg,degree,fit_lower,k", CLASS_CASES)
def test_column_classes_every_dispatch(reg, degree, fit_lower, k, monkeypatch):
    """Singles, short columns of 2 / 8, single chunks of 9..64 (flagged), split columns of 65 / 128 / 129 and 256
    nonzeros in every minibatch, for every (G, KCH) of launch_minibatch (k <= 8, 16, 32, 64, 128) and NORD 1 / 3."""
    plans = _capture_plans(monkeypatch)
    X, y = _class_problem()
    kw = _kw(regularizer=reg, degree=degree, fit_lower=fit_lower, n_components=k)
    out = _oracle_fit("classes", X, y, kw)
    est = _fit_twice(kw, X, y)
    counts = _assert_classes(plans[0], range(4))
    assert plans[0].n_minibatches == 5 and np.diff(plans[0].mb_eptr)[-1] > 0
    err, _ = _compare(est, out, X, y, check_objective=False)
    print(reg, degree, fit_lower, k, "classes (singles, short, chunks, flagged, multi) per minibatch", counts,
          "err", err, "nonzero fraction", _nonzero_fraction(est))


EDGES = ["empty_minibatches", "batch_size_1", "batch_size_above_n", "shuffle", "build_groups"]


@pytest.mark.parametrize("reg", ["l1", "squaredl12"])
@pytest.mark.parametrize("edge", EDGES)
def test_minibatch_edges(edge, reg, monkeypatch):
    """Minibatches without nonzeros (the cols launches are skipped, the rows pass, statistics and selection still
    run), batch_size=1, one minibatch shorter than batch_size, three reshuffled epochs, a plan built in groups."""
    plans = _capture_plans(monkeypatch, group_entries=700 if edge == "build_groups" else None)
    kw = _kw(regularizer=reg, n_components=5, degree=3, fit_lower="explicit")
    if edge == "empty_minibatches":
        X, y = _class_problem(n_mb=5, empty=(1, 3))
    elif edge == "batch_size_1":
        from sparsepoly_b200 import synth
        X = synth.uniform_sparse(300, 40, 4, 3)
        y = _labels(300, 4)
        kw.update(batch_size=1, max_iter=3, gamma=1e-5)
    elif edge == "batch_size_above_n":
        X, y = _class_problem(n_mb=2, tail=60)
        kw.update(batch_size=5000, max_iter=4)
    elif edge == "shuffle":
        X, y = _class_problem()
        kw.update(shuffle=True, max_iter=3)
    else:
        X, y = _class_problem()
    out = _oracle_fit(edge, X, y, kw)
    est = _fit_twice(kw, X, y)
    p = plans[0]
    eptr = np.diff(p.mb_eptr)
    if edge == "empty_minibatches":
        assert eptr[1] == 0 and eptr[3] == 0 and np.all(eptr[[0, 2, 4, 5]] > 0), eptr
        _assert_classes(p, (0, 2, 4))
    elif edge == "batch_size_1":
        assert p.n_minibatches == 300 and p.max_cols <= 4 and p.n_cols == X.nnz
    elif edge == "batch_size_above_n":
        assert p.n_minibatches == 1 and p.batch_local == 5000 and eptr[0] == X.nnz
    elif edge == "shuffle":
        assert len(plans) == 2 * (1 + kw["max_iter"])      # the setup's plan and one per epoch, two fits
        orders = [q.e_pos.cpu().numpy() for q in plans[1:4]]
        assert not np.array_equal(orders[0], orders[1]) and not np.array_equal(orders[1], orders[2])
    else:
        full = _plans_equal_default(p, X)
        assert full, "the grouped plan differs from the one-group plan"
        _assert_classes(p, range(4))
    err, _ = _compare(est, out, X, y, check_objective=False)
    print(edge, reg, "minibatches", p.n_minibatches, "entries per minibatch", eptr.tolist()[:8], "err", err,
          "nonzero fraction", _nonzero_fraction(est))


def _plans_equal_default(p, X):
    """A plan built in groups of 700 entries (one or two minibatches per group) equals the one-group plan."""
    import torch
    from sparsepoly_b200.psgd_plan import PsgdPlan
    from sparsepoly_b200.dataset import DeviceDataset
    ds = DeviceDataset(X, need_csr=True, need_csc=False)
    q = PsgdPlan(ds.csr, torch.arange(X.shape[0], dtype=torch.int32, device="cuda"), X.shape[1], p.batch_local)
    names = ("e_pos", "e_x", "u_feat", "u_ptr", "sg_u", "sc_ptr", "sc_u", "lc_u", "lc_e0", "lc_cnt", "ml_u", "ml_c0")
    host = ("mb_eptr", "mb_uptr", "mb_sgptr", "mb_shptr", "mb_lcptr", "mb_mlptr")
    return (all(torch.equal(getattr(p, a), getattr(q, a)) for a in names)
            and all(np.array_equal(getattr(p, a), getattr(q, a)) for a in host))


# ============================================================================ b. squared-l1,2 selection paths
def _selection(est):
    s = est._psgd_stats["selection"]
    calls, band, generic, half = int(s["prox_calls"]), int(s["band_solves"]), int(s["generic_solves"]), s["band_half_width"]
    assert band + generic == calls
    return calls, band, generic, half


def _stats_problem(d, seed=0):
    """A few hundred rows touching the first 30 features of d; the selection sees every row of P."""
    from sparsepoly_b200 import synth
    X = synth.uniform_sparse(400, 30, 4, seed)
    X = sp.csr_matrix((X.data, X.indices, X.indptr), shape=(400, d))
    return X, _labels(400, seed + 1)


# (k, degree, fit_lower, d): VEC = 2 (even k) and 1 (odd k); one order and two; d below one statistics block
# (256 / (k / VEC) rows) and above STAT_PART_MAX = 444 blocks of them
HIT_CASES = [(4, 2, None, 40), (5, 2, None, 40), (4, 3, "explicit", 40), (5, 3, "explicit", 40),
             (2, 2, None, 200_000), (3, 2, None, 200_000), (6, 3, "explicit", 200_000)]


@pytest.mark.parametrize("k,degree,fit_lower,d", HIT_CASES)
def test_selection_band_hit(k, degree, fit_lower, d):
    """A slowly moving threshold (small steps, constant rate): after the first call (generic passes: no
    prediction yet) the threshold lands in the predicted band and the exact band sums solve it."""
    X, y = _stats_problem(d)
    rng = np.random.RandomState(1)
    n_orders = degree - 1 if fit_lower == "explicit" else 1
    P_init = 0.01 * rng.randn(n_orders, k, d)
    kw = _kw(n_components=k, degree=degree, fit_lower=fit_lower, eta0=0.01, gamma=0.5 / d, batch_size=40,
             max_iter=2)
    out = _oracle_fit("hit", X, y, kw, P_init=P_init)
    est = _fit_twice(kw, X, y, P_init=P_init)
    calls, band, generic, half = _selection(est)
    print("hit", k, degree, fit_lower, d, "calls", calls, "band", band, "generic", generic, "half-width", half)
    assert calls == 20 and band >= calls - 2 and generic <= 2, (calls, band, generic)
    _compare(est, out, X, y, check_objective=False)
    _nonzero_fraction(est)


@pytest.mark.parametrize("lr,power_t,reg_strength", [("invscaling", 5.0, 1e-2), ("pegasos", 1.0, 10.0),
                                                     ("optimal", 1.0, 1e-2)])
def test_selection_band_miss(lr, power_t, reg_strength):
    """Strength jumps: invscaling with power_t = 5 divides the step by 32 after the first minibatch and the
    predicted threshold (clamped to half the last one) misses; pegasos / optimal change the strength fast early
    on.  A miss takes the generic passes and doubles the half-width (up to 0.1)."""
    X, y = _stats_problem(60)
    P_init = 0.01 * np.random.RandomState(2).randn(1, 4, 60)
    kw = _kw(n_components=4, learning_rate=lr, power_t=power_t, eta0=1.0, alpha=reg_strength, beta=reg_strength,
             gamma=2e-3,
             batch_size=40, max_iter=2)
    out = _oracle_fit("miss", X, y, kw, P_init=P_init)
    est = _fit_twice(kw, X, y, P_init=P_init)
    calls, band, generic, half = _selection(est)
    print("miss", lr, power_t, "calls", calls, "band", band, "generic", generic, "half-width", half)
    if lr == "invscaling":
        assert generic >= 3 and half > 0.02, (generic, half)
    else:
        assert generic >= 1 and band + generic == calls
    _compare(est, out, X, y, check_objective=False)


@pytest.mark.parametrize("d", [2_000_000])
def test_selection_band_overflow(d):
    """Column 0 of P holds d values spread evenly over (0, 1], in feature order (the band's members sit in
    consecutive rows: every statistics block that holds them spills its BAND_BLK staging slots into the global
    reservation), with strength 1 / d: thousands of values fall inside every band.  The band overflows
    SP_PSGD_BAND_CAP, the generic passes solve, and the half-width halves -- it only shrinks on an overflow --
    while the model still matches the oracle."""
    rng = np.random.RandomState(3)
    X = sp.csr_matrix((rng.uniform(0.2, 1.0, 12), (np.repeat(np.arange(4), 3), rng.choice(20, 12))), shape=(4, d))
    X.sum_duplicates()
    X.sort_indices()
    y = np.array([1.0, -1.0, 1.0, -1.0])
    P_init = np.empty((1, 2, d))
    P_init[0, 0] = np.arange(1, d + 1) / d
    P_init[0, 1] = 0.01 * rng.randn(d)
    kw = _kw(n_components=2, eta0=0.1, alpha=0.0, beta=0.0, gamma=10.0 / d, batch_size=1, max_iter=1)
    out = _oracle_fit("overflow", X, y, kw, P_init=P_init)
    est = _fit_twice(kw, X, y, P_init=P_init)
    calls, band, generic, half = _selection(est)
    s = est._psgd_stats["selection"]
    print("overflow d", d, "calls", calls, "band", band, "generic", generic, "half-width", half, "stats", s)
    assert calls == 4 and generic >= 3 and half < 0.02, (calls, generic, half)
    _compare(est, out, X, y, check_objective=False)
    assert 0.05 < np.mean(out["P_"][0, 0] != 0) < 0.95


# ============================================================================ c. long horizons of the lazy frame
def _frames_expected(factors_C, factors_Cw, calls):
    """(C, Cw) after every call of the fold rule replayed on the host: `calls` = minibatches per call."""
    C = Cw = 1.0
    out, t, folds = [], 0, []
    for n_mb in calls:
        for _ in range(n_mb):
            C, Cw = C * factors_C[t], Cw * factors_Cw[t]
            t += 1
            if not (1e-100 < C < 1e100 and 1e-100 < Cw < 1e100):
                C = Cw = 1.0
                folds.append(t)
        out.append((C, Cw))
    return out, folds


@pytest.mark.parametrize("reg", ["l1", "squaredl12"])
@pytest.mark.parametrize("batch_size", [1, 3, 8])
def test_beta_zero_long_horizon(reg, batch_size, monkeypatch):
    """beta = 0: C stays 1 while the thresholds grow without bound over several epochs of small minibatches."""
    from sparsepoly_b200 import synth
    frames = _record_frames(monkeypatch)
    n = 600
    X = synth.uniform_sparse(n, 50, 4, 8)
    y = _labels(n, 9)
    kw = _kw(regularizer=reg, n_components=4, beta=0.0, alpha=1e-3, gamma=2e-4, eta0=0.05, batch_size=batch_size,
             max_iter=4)
    out = _oracle_fit("beta0", X, y, kw)
    est = _fit_twice(kw, X, y)
    assert all(C == 1.0 for C, _ in frames), frames
    print("beta=0", reg, batch_size, "minibatches", 4 * -(-n // batch_size), "final (C, Cw)", frames[-1])
    _compare(est, out, X, y, check_objective=False)
    _nonzero_fraction(est)


F_C, F_CW = 1.0 + 0.5 * 0.02, 1.0 + 0.5 * 1.0          # per-minibatch growth of C / Cw in _overflow_kw


def _overflow_problem(n):
    """batch_size=1 and eta * alpha = 0.5: Cw grows by 1.5 per minibatch (past 1e100 after 568, inf after ~1750)
    while w itself stays O(1); C grows by 1.01."""
    from sparsepoly_b200 import synth
    X = synth.uniform_sparse(n, 40, 5, 11)
    return X, _labels(n, 5)


def _overflow_kw(reg, **extra):
    kw = _kw(regularizer=reg, n_components=4, alpha=1.0, beta=0.02, gamma=1e-4, eta0=0.5, batch_size=1, max_iter=1)
    kw.update(extra)
    return kw


@pytest.mark.parametrize("reg", ["l1", "squaredl12"])
def test_frame_folds_at_epoch_ends(reg, monkeypatch):
    """568 minibatches per epoch, eta * alpha = 0.5: Cw passes 1e100 at the last minibatch of every epoch.  A callback syncs after
    every epoch (the frame is materialised and the scales reset), and the model of every epoch matches the
    oracle's fit of that many epochs."""
    frames = _record_frames(monkeypatch)
    n = 568
    X, y = _overflow_problem(n)
    seen = []
    kw = _overflow_kw(reg, max_iter=3, eta0=0.1, alpha=5.0, gamma=1e-5)     # (small steps: three epochs stay well conditioned)
    est = _fm_estimator(kw)
    est.set_params(callback=lambda e: seen.append((e.P_.copy(), e.w_.copy())), n_calls=1)
    _fit(est, X, y)
    assert 1.5 ** 567 < 1e100 < 1.5 ** 568
    want, folds = _frames_expected([1.0 + 0.1 * 0.02] * 3 * n, [1.0 + 0.1 * 5.0] * 3 * n, [n] * 3)
    assert folds == [n, 2 * n, 3 * n]
    assert frames == [(1.0, 1.0)] * 3, frames
    assert len(seen) == 3
    for e, (P, w) in enumerate(seen):
        out = _oracle_fit("epoch_end", X, y, dict(kw, max_iter=e + 1))
        assert rel_err(P, out["P_"]) <= 1e-9 and rel_err(w, out["w_"]) <= 1e-9, e
    _compare(est, _oracle_fit("epoch_end", X, y, kw), X, y, check_objective=False)
    print("epoch-end folds", reg, "folds after minibatch", folds, "(C, Cw) after every epoch", frames)


@pytest.mark.parametrize("reg", ["l1", "squaredl12"])
def test_frame_folds_inside_an_epoch(reg, monkeypatch):
    """2000 minibatches in one epoch: Cw would overflow to inf after ~1750 (w then reads back as 0); the run folds
    the frame after minibatches 568, 1136 and 1704 and ends at the oracle's model."""
    frames = _record_frames(monkeypatch)
    n = 2000
    X, y = _overflow_problem(n)
    kw = _overflow_kw(reg)
    out = _oracle_fit("inside", X, y, kw)
    est = _fit_twice(kw, X, y)
    want, folds = _frames_expected([F_C] * n, [F_CW] * n, [n])
    assert folds == [568, 1136, 1704] and frames[0] == want[0], (frames, want)
    assert np.max(np.abs(out["w_"])) > 1e-2
    print("inside-epoch folds", reg, folds, "final (C, Cw)", frames[0])
    _compare(est, out, X, y, check_objective=False)


def test_frame_folds_inside_a_long_epoch_of_small_values(monkeypatch):
    """8000 minibatches of one row, eta * beta = 0.1: C = 1.1^8000 ~ 1e331 would overflow; the model keeps most of
    P nonzero at ~1e-281 (normal numbers), so a frame read as 0 fails both the error and the support check."""
    from sparsepoly_b200 import synth
    frames = _record_frames(monkeypatch)
    n = 8000
    X = synth.uniform_sparse(n, 40, 5, 11)
    y = _labels(n, 5)
    kw = _kw(n_components=4, alpha=0.0, beta=0.2, gamma=1e-4, eta0=0.5, batch_size=1, max_iter=1)
    out = _oracle_fit("issue", X, y, kw)
    est = _fit_twice(kw, X, y)
    want, folds = _frames_expected([1.0 + 0.5 * 0.2] * n, [1.0] * n, [n])
    assert len(folds) == 3 and frames[0] == want[0], (folds, frames, want)
    assert np.mean(out["P_"] != 0) > 0.5 and np.max(np.abs(out["P_"])) > 1e-290
    print("small-value folds", folds, "final (C, Cw)", frames[0], "max |P|", np.max(np.abs(out["P_"])))
    _compare(est, out, X, y, check_objective=False)


@pytest.mark.parametrize("reg", ["l1", "squaredl12"])
def test_frame_folds_across_partial_fit_calls(reg, monkeypatch):
    """The same 2000 minibatches as chunks of 300 rows (the last one 200): the folds fall inside calls and the
    model after the last call equals fit's bit for bit; the scales after every call follow the fold rule."""
    frames = _record_frames(monkeypatch)
    n = 2000
    X, y = _overflow_problem(n)
    kw = _overflow_kw(reg)
    fit = _fit(_fm_estimator(kw), X, y)
    del frames[:]
    est = _fm_estimator(kw)
    bounds = list(range(0, n, 300)) + [n]
    for a, b in zip(bounds[:-1], bounds[1:]):
        est.partial_fit(X[a:b], y[a:b], classes=np.array([-1.0, 1.0]))
    want, folds = _frames_expected([F_C] * n, [F_CW] * n, np.diff(bounds).tolist())
    assert frames == want, (frames, want)
    assert np.array_equal(est.P_, fit.P_) and np.array_equal(est.w_, fit.w_)
    assert est.it_ == fit.it_ == n + 1
    out = _oracle_fit("inside", X, y, kw)
    assert rel_err(est.P_, out["P_"]) <= 1e-9 and rel_err(est.w_, out["w_"]) <= 1e-9
    print("partial_fit folds", reg, folds, "(C, Cw) after every call", frames)
