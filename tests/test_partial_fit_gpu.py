"""partial_fit of the psgd factorization machines: chunks of rows streamed from the host, one psgd pass per call.

  * chunks of a multiple of batch_size rows, in order, E times = fit(max_iter=E) on their concatenation, bit for bit
    (planned path: l1 / squaredl12), which also shows that the per-call read-out leaves the lazy frame alone;
  * ragged chunks and the dense-gradient path (l21 / squaredl21) against the oracle driven call by call, 1e-9;
  * sp_psgd_plan_read against materialise + transpose, bit for bit, with the context unchanged;
  * shuffle, continuation after fit / pickle, the classifier's labels, and device memory over many calls."""
import pickle
import warnings

import numpy as np
import pytest

from golden_util import rel_err, same_support

pytestmark = pytest.mark.gpu

TOL = 1e-9
B = 128


def _problem(n, d, seed, clf):
    from sparsepoly_b200 import synth
    X = synth.criteo_like(n, d, seed)
    rng = np.random.RandomState(seed + 1)
    y = np.where(rng.rand(n) < 0.3, 1.0, -1.0) if clf else rng.randn(n)
    return X, y


def _kw(reg, degree=2, k=8, clf=True, **extra):
    kw = dict(degree=degree, loss="logistic" if clf else "squared", n_components=k, solver="psgd", regularizer=reg,
              alpha=1e-3, beta=1e-3, gamma=1e-3 if reg in ("l1", "l21") else 3e-3, eta0=0.1, batch_size=B,
              fit_lower="explicit", tol=-1.0, n_iter_no_change=10 ** 9, random_state=0)
    kw.update(extra)
    return kw


def _est(kw):
    import sparsepoly_b200 as S
    if kw["loss"] == "squared":
        return S.SparseFactorizationMachineRegressor(**{k: v for k, v in kw.items() if k != "loss"})
    return S.SparseFactorizationMachineClassifier(**kw)


def _clf_est(kw):
    import sparsepoly_b200 as S
    return S.SparseFactorizationMachineClassifier(**kw)


def _bounds(sizes):
    b = np.concatenate([[0], np.cumsum(sizes)])
    return list(zip(b[:-1], b[1:]))


def _stream(est, X, y, sizes, passes=1, classes=None):
    for _ in range(passes):
        for a, b in _bounds(sizes):
            est.partial_fit(X[a:b], y[a:b], classes=classes)
    return est


def _fit(est, X, y):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return est.fit(X, y)


def _oracle_calls(kw, X, y, sizes, passes=1, P=None, w=None, lams=None, it=1, check=None):
    """The oracle driven call by call: one max_iter=1 fit per chunk from the previous call's model."""
    from oracle import oracle as O
    okw = {k: v for k, v in kw.items() if k not in ("solver", "tol", "n_iter_no_change", "max_iter")}
    for _ in range(passes):
        for a, b in _bounds(sizes):
            out = O.fit_fm(X[a:b], y[a:b], solver="psgd", max_iter=1, tol=-1.0, n_iter_no_change=10 ** 9,
                           P_init=P, w_init=w, lams_init=lams, it_init=it, **okw)
            P, w, lams, it = out["P_"], out["w_"], out["lams_"], out["it_"]
            if check is not None:
                check(P, w, it)
    return P, w, lams, it


def _assert_close(est, P, w, it):
    assert rel_err(est.P_, P) <= TOL and same_support(est.P_, P)
    assert rel_err(est.w_, w) <= TOL
    assert est.it_ == it


# ------------------------------------------------------------------------------------------------ chunked == fit
BITWISE = [("l1", 2, 8, False), ("squaredl12", 2, 32, True), ("l1", 3, 128, True), ("squaredl12", 3, 8, False),
           ("squaredl12", 2, 128, False)]


@pytest.mark.parametrize("passes", [1, 2])
@pytest.mark.parametrize("reg,degree,k,clf", BITWISE, ids=[f"{c[0]}-deg{c[1]}-k{c[2]}-{'clf' if c[3] else 'reg'}"
                                                           for c in BITWISE])
def test_chunks_equal_fit_bit_for_bit(reg, degree, k, clf, passes):
    sizes = [3 * B, 5 * B, 2 * B]
    X, y = _problem(sum(sizes), 900, 3, clf)
    kw = _kw(reg, degree, k, clf)
    full = _fit(_est(dict(kw, max_iter=passes)), X, y)
    est = _stream(_est(kw), X, y, sizes, passes, classes=[-1.0, 1.0] if clf else None)
    assert np.array_equal(est.P_, full.P_) and np.array_equal(est.w_, full.w_)
    assert np.array_equal(est.lams_, full.lams_) and est.it_ == full.it_
    assert est.n_iter_ == 3 * passes and np.mean(est.P_ != 0) < 1.0       # (the prox did zero entries)


# ------------------------------------------------------------------------------ ragged chunks, dense path, oracle
@pytest.mark.parametrize("reg", ["l1", "squaredl12", "l21", "squaredl21"])
def test_ragged_chunks_match_oracle_call_by_call(reg):
    sizes = [250, 130, 400, 77]                       # not multiples of batch_size; the third is larger than the first
    X, y = _problem(sum(sizes), 700, 5, True)
    kw = _kw(reg, 2, 8, True, batch_size=100)
    est = _clf_est(kw)
    calls = iter(_bounds(sizes))

    def check(P, w, it):
        a, b = next(calls)
        est.partial_fit(X[a:b], y[a:b], classes=[-1.0, 1.0])
        _assert_close(est, P, w, it)
    _oracle_calls(kw, X, y, sizes, check=check)
    assert est.n_iter_ == len(sizes)


# ------------------------------------------------------------------------------------- the non-mutating read-out
@pytest.mark.parametrize("n_orders", [1, 2, 3, 4])
@pytest.mark.parametrize("k", [1, 7, 63, 128])
def test_plan_read_equals_materialise_and_transpose(k, n_orders):
    import torch

    from sparsepoly_b200 import solvers
    X, y = _problem(6 * 64, 500, 7, True)
    est = _clf_est(_kw("l1", n_orders + 1, k, True, batch_size=64, gamma=1e-2))
    est.partial_fit(X, y, classes=[-1.0, 1.0])
    ctx = est._psgd_stream["ctx"]
    assert ctx.struct.C != 1.0 and ctx.struct.Cw != 1.0 and bool((ctx.thr > 0).all())
    before = (ctx.P.clone(), ctx.w.clone(), ctx.thr.clone(), ctx.struct.C, ctx.struct.Cw)
    d = X.shape[1]
    P_out = torch.empty((n_orders, k, d), dtype=torch.float64, device=ctx.P.device)
    w_out = torch.empty(d, dtype=torch.float64, device=ctx.P.device)
    solvers.psgd_planned_read(ctx, P_out, w_out)
    torch.cuda.synchronize()
    assert torch.equal(ctx.P, before[0]) and torch.equal(ctx.w, before[1]) and torch.equal(ctx.thr, before[2])
    assert (ctx.struct.C, ctx.struct.Cw) == before[3:]
    assert np.array_equal(P_out.cpu().numpy(), est.P_) and np.array_equal(w_out.cpu().numpy(), est.w_)
    P = torch.empty((n_orders, d, k), dtype=torch.float64, device=ctx.P.device)
    w = torch.empty(d, dtype=torch.float64, device=ctx.P.device)
    solvers.psgd_planned_end(ctx, 0, None, True)
    ctx.store_model(P, w)
    P_ref = torch.stack([solvers.transpose(P[o]) for o in range(n_orders)])
    assert torch.equal(P_out, P_ref) and torch.equal(w_out, w)
    assert bool((P_ref == 0).any()) and bool((P_ref != 0).any())


# --------------------------------------------------------------------------------------------------- shuffle
def test_shuffle_one_call_equals_fit_and_three_calls_match_oracle():
    from oracle import oracle as O
    sizes = [3 * B, 2 * B + 31, 4 * B]
    X, y = _problem(sum(sizes), 800, 11, True)
    kw = _kw("squaredl12", 2, 16, True, shuffle=True)
    a, b = _bounds(sizes)[0]
    full = _fit(_clf_est(dict(kw, max_iter=1)), X[a:b], y[a:b])
    one = _clf_est(kw).partial_fit(X[a:b], y[a:b], classes=[-1.0, 1.0])
    assert np.array_equal(one.P_, full.P_) and np.array_equal(one.w_, full.w_) and one.it_ == full.it_
    # the oracle fed the same draws: the initial model, then one permutation of every chunk from one generator
    est = _stream(_clf_est(kw), X, y, sizes, classes=[-1.0, 1.0])
    rng = np.random.RandomState(0)
    P = 0.01 * rng.randn(1, 16, X.shape[1])
    w, lams, it = np.zeros(X.shape[1]), np.ones(16), 1
    okw = {k: v for k, v in kw.items() if k not in ("solver", "tol", "n_iter_no_change", "shuffle")}
    for a, b in _bounds(sizes):
        order = np.arange(b - a, dtype=np.int32)
        rng.shuffle(order)
        out = O.fit_fm(X[a:b][order], y[a:b][order], solver="psgd", max_iter=1, tol=-1.0, n_iter_no_change=10 ** 9,
                       P_init=P, w_init=w, lams_init=lams, it_init=it, **okw)
        P, w, lams, it = out["P_"], out["w_"], out["lams_"], out["it_"]
    _assert_close(est, P, w, it)


# ------------------------------------------------------------------------------- continuation and interaction
def test_fit_then_partial_fit_continues_from_the_fitted_model():
    X, y = _problem(1500, 800, 13, False)
    kw = _kw("l1", 3, 8, False)
    est = _fit(_est(dict(kw, max_iter=2)), X[:1000], y[:1000])
    P0, w0, lams0, it0 = est.P_.copy(), est.w_.copy(), est.lams_.copy(), est.it_
    est.partial_fit(X[1000:], y[1000:])
    assert est.n_iter_ == 1
    P, w, _, it = _oracle_calls(kw, X[1000:], y[1000:], [500], P=P0, w=w0, lams=lams0, it=it0)
    _assert_close(est, P, w, it)


def test_fit_after_partial_fit_is_a_fresh_fit():
    X, y = _problem(1200, 800, 17, True)
    kw = _kw("squaredl12", 2, 8, True, max_iter=2)
    est = _stream(_clf_est(kw), X, y, [400, 400], classes=[-1.0, 1.0])
    _fit(est, X, y)
    fresh = _fit(_clf_est(kw), X, y)
    assert np.array_equal(est.P_, fresh.P_) and np.array_equal(est.w_, fresh.w_) and est.it_ == fresh.it_
    assert not hasattr(est, "_psgd_stream") and not hasattr(est, "batch_size_")


@pytest.mark.parametrize("reg", ["squaredl12", "l21"])
def test_pickle_mid_stream_then_continue(reg):
    sizes = [300, 256, 410]
    X, y = _problem(sum(sizes), 700, 19, True)
    kw = _kw(reg, 2, 8, True, batch_size=90)
    est = _clf_est(kw)
    bounds = _bounds(sizes)
    for a, b in bounds[:2]:
        est.partial_fit(X[a:b], y[a:b], classes=[-1.0, 1.0])
    est = pickle.loads(pickle.dumps(est))
    assert not hasattr(est, "_psgd_stream")
    a, b = bounds[2]
    est.partial_fit(X[a:b], y[a:b])
    assert est.n_iter_ == 3
    P, w, _, it = _oracle_calls(kw, X, y, sizes)
    _assert_close(est, P, w, it)


def test_auto_batch_size_is_resolved_once():
    X, y = _problem(900, 800, 23, True)
    X2 = X[600:].copy()
    X2.data[::3] = 0.0
    X2.eliminate_zeros()                                      # other density: "auto" would resolve differently
    X1 = X[:600]
    kw = _kw("l1", 2, 8, True, batch_size="auto")
    est = _clf_est(kw)
    est.partial_fit(X1, y[:600], classes=[-1.0, 1.0])
    bs = int(X1.shape[0] * X1.shape[1] / X1.nnz)
    assert est.batch_size_ == bs and int(X2.shape[0] * X2.shape[1] / X2.nnz) != bs
    est.partial_fit(X2, y[600:])
    assert est.batch_size_ == bs
    okw = dict(kw, batch_size=bs)
    P, w, lams, it = _oracle_calls(okw, X1, y[:600], [600])
    P, w, _, it = _oracle_calls(okw, X2, y[600:], [300], P=P, w=w, lams=lams, it=it)
    _assert_close(est, P, w, it)


# ------------------------------------------------------------------------------------------- classifier labels
def test_classifier_labels():
    sizes = [3 * B, 2 * B, 2 * B]
    X, y = _problem(sum(sizes), 800, 29, True)
    y[sizes[0]:sizes[0] + sizes[1]] = 1.0                    # the second chunk holds one class only
    names = np.where(y > 0, "pos", "neg")
    kw = _kw("squaredl12", 2, 8, True)
    with pytest.raises(ValueError, match="classes"):
        _clf_est(kw).partial_fit(X[:B], names[:B])
    est = _stream(_clf_est(kw), X, names, sizes, classes=["neg", "pos"])
    ref = _stream(_clf_est(kw), X, y, sizes, classes=[-1.0, 1.0])
    assert np.array_equal(est.P_, ref.P_) and np.array_equal(est.w_, ref.w_)
    pred = est.predict(X[:200])
    assert pred.dtype == names.dtype and set(pred) <= {"neg", "pos"}
    assert np.array_equal(pred == "pos", ref.predict(X[:200]) == 1.0)
    bad = names[:B].copy()
    bad[5] = "other"
    with pytest.raises(ValueError, match="not in classes"):
        est.partial_fit(X[:B], bad)
    assert est.n_iter_ == len(sizes)


# ------------------------------------------------------------------------------------------------------ memory
@pytest.mark.parametrize("reg", ["squaredl12", "l21"])
def test_device_memory_does_not_grow_with_calls(reg):
    import torch
    X, y = _problem(2 * 500, 1200, 31, True)
    est = _clf_est(_kw(reg, 2, 16, True))
    after = {}
    for c in range(20):                          # two chunks of equal shape in turn: the scratch has seen both by call 2
        a = (c % 2) * 500
        est.partial_fit(X[a:a + 500], y[a:a + 500], classes=[-1.0, 1.0])
        torch.cuda.synchronize()
        after[c + 1] = torch.cuda.memory_allocated()
    assert after[20] == after[2], after
