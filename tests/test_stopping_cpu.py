"""Stopping parameters chosen from a per-epoch trace, and the oracle's stop bookkeeping.

A fit stops on one value per epoch: the violation sum of pcd / pbcd (`viol < tol`) or psgd's mean epoch loss (the
plateau rule: an epoch counts as no improvement when `loss > best - tol`; n_iter_no_change such epochs in a row
stop the fit).  tests/test_stopping_gpu.py fits the device with parameters that the helpers below choose from the
oracle's tol=-1 trace, so that the device and the oracle must stop at one chosen epoch.  Each decision on the way
is taken with a relative margin of at least MARGIN: a 1e-12 difference of a traced value cannot flip it, so a
stop at another epoch is a wrong value, not rounding.

Here the helpers are checked on their own: replayed by hand over synthetic traces, refusing traces with no safe
choice, and against oracle.fit_fm / fit_all_subsets, whose n_iter_ is the index of the last epoch run and whose
converged flag says whether the rule (not max_iter) ended the fit."""
import math
import re

import numpy as np
import pytest

MARGIN = 1e-6         # smallest relative margin of a stopping decision the chosen parameters may leave
DROP = 1e-3           # a violation counts as a new minimum when 0.1 % below every earlier one

_LINE = re.compile(r"^(Iteration|Epoch|Call) (\d+) (?:violation sum|loss) (\S+)$", re.M)


# ------------------------------------------------------------------------------------------------ the device trace
def parse_traces(text):
    """The per-epoch values of the verbose lines in `text` ("Iteration i violation sum v" of pcd / pbcd /
    all-subsets, "Epoch i loss v" of psgd, "Call i loss v" of partial_fit), one list per fit: a line numbered 1
    starts the next fit (fit_many prints its models one after the other).  Python prints a float's round-trip
    repr, so each value is exactly the one the stopping rule compared."""
    traces = []
    for _, i, v in _LINE.findall(text):
        i = int(i)
        if i == 1:
            traces.append([])
        assert traces and i == len(traces[-1]) + 1, f"verbose lines out of order at {i}"
        traces[-1].append(float(v))
    return traces


# --------------------------------------------------------------------------------------------- violation sum < tol
def replay_viol(trace, tol):
    """(n_iter_, converged) of `viol < tol` over the epochs of `trace` (max_iter = len(trace))."""
    for i, v in enumerate(trace):
        if v < tol:
            return i, True
    return len(trace) - 1, False


def viol_margin(trace, tol, stop):
    """Smallest relative distance between tol and the violations it was compared with (epochs 0..stop)."""
    return min(abs(v - tol) / tol for v in trace[:stop + 1])


def first_drop(trace):
    """The first epoch e >= 1 whose violation is below every earlier one by at least DROP."""
    for e in range(1, len(trace)):
        if trace[e] < (1.0 - DROP) * min(trace[:e]):
            return e
    raise ValueError(f"no epoch of {trace} drops below the earlier ones by {DROP}")


def tol_stopping_at(trace, e):
    """(tol, margin): a tol with which `viol < tol` stops after epoch e.  e = 0: just above trace[0]; e >= 1: the
    geometric mean of trace[e] and the smallest earlier violation, which trace[e] must undercut by DROP."""
    if e == 0:
        tol = trace[0] * (1.0 + DROP)
    else:
        prev = min(trace[:e])
        if not trace[e] < (1.0 - DROP) * prev:
            raise ValueError(f"epoch {e} ({trace[e]!r}) does not undercut the earlier minimum {prev!r} by {DROP}")
        tol = math.sqrt(trace[e] * prev)
    if not tol > 0.0:
        raise ValueError(f"no positive tol stops at epoch {e} of {trace}")
    margin = viol_margin(trace, tol, e)
    assert replay_viol(trace, tol) == (e, True) and margin >= MARGIN, (trace, e, tol, margin)
    return tol, margin


def tol_never(trace):
    """(tol, margin): half the smallest violation; no epoch stops."""
    if not min(trace) > 0.0:
        raise ValueError(f"a zero violation in {trace}: every positive tol stops there")
    tol = min(trace) / 2
    return tol, viol_margin(trace, tol, len(trace) - 1)


# ------------------------------------------------------------------------------------------- psgd's plateau rule
def replay_plateau(trace, tol, n_iter_no_change):
    """(n_iter_, converged, resets) of the plateau rule over the epoch losses of `trace` (max_iter = len(trace));
    resets counts the epochs that set a running no-improvement count back to zero."""
    no_improve, best, resets = 0, np.inf, 0
    for i, loss in enumerate(trace):
        if loss > best - tol:
            no_improve += 1
        else:
            resets += no_improve > 0
            no_improve = 0
        best = min(best, loss)
        if no_improve >= n_iter_no_change:
            return i, True, resets
    return len(trace) - 1, False, resets


def plateau_critical(trace):
    """best_{i-1} - L_i for the epochs i >= 1: epoch i counts as no improvement exactly when tol exceeds it (epoch 0
    never does: best is inf).  The running best does not depend on tol."""
    best, out = np.inf, []
    for i, loss in enumerate(trace):
        if i > 0:
            out.append(best - loss)
        best = min(best, loss)
    return out


def plateau_margin(trace, tol, stop):
    """Smallest distance, relative to the loss compared, between tol and the critical values of epochs 1..stop."""
    crit = plateau_critical(trace)
    return min((abs(tol - crit[i - 1]) / abs(trace[i]) for i in range(1, stop + 1)), default=np.inf)


def choose_plateau_tol(trace, n_iter_no_change):
    """(tol, stop, margin, resets): tol at the middle of the widest gap between two adjacent critical values whose
    replay stops before the trace ends, preferring gaps whose replay also resets the no-improvement count.  A tol
    outside every critical value takes all decisions one way; the gaps between them are where a wrong loss changes
    the stop epoch.  Refuses (ValueError) when that gap leaves a decision closer than MARGIN, as ties do."""
    crit = sorted(set(plateau_critical(trace)))
    best = None
    for lo, hi in zip(crit[:-1], crit[1:]):
        tol = 0.5 * (lo + hi)
        stop, converged, resets = replay_plateau(trace, tol, n_iter_no_change)
        key = (resets > 0, hi - lo)
        if converged and stop < len(trace) - 1 and (best is None or key > best[0]):
            best = (key, tol, stop, resets)
    if best is None:
        raise ValueError(f"no tol stops {trace} with n_iter_no_change={n_iter_no_change} before its last epoch")
    _, tol, stop, resets = best
    margin = plateau_margin(trace, tol, stop)
    if margin < MARGIN:
        raise ValueError(f"the widest gap leaves a margin of {margin:.2e} < {MARGIN}")
    return tol, stop, margin, resets


# ============================================================================================== tests of the helpers
def test_parse_traces_splits_fits_and_round_trips():
    vals = [0.1, 1 / 3, 2.5e-17, 123456.789e10]
    text = "".join(f"Iteration {i + 1} violation sum {v}\n" for i, v in enumerate(vals))
    text += "Converged at iteration 4\nIteration 1 violation sum 7.0\n"
    text += "Epoch 1 loss 0.6931471805599453\nEpoch 2 loss 0.5\nCall 1 loss 0.25\n"
    got = parse_traces(text)
    assert got == [vals, [7.0], [0.6931471805599453, 0.5], [0.25]]
    assert all(float(repr(v)) == v for v in vals)
    with pytest.raises(AssertionError):
        parse_traces("Iteration 2 violation sum 1.0\n")


def _by_hand_viol(trace, tol):
    for i, v in enumerate(trace):
        if v < tol:
            return i
    return None


@pytest.mark.parametrize("trace", [[5.0, 3.0, 2.9, 1.0, 0.5], [1.0, 2.0, 0.999, 0.5, 0.1], [4.0, 4.0, 4.0, 3.0]])
def test_viol_tol_choices_stop_where_replayed(trace):
    e = first_drop(trace)
    assert all(trace[e] < (1 - DROP) * v for v in trace[:e])
    assert all(not trace[i] < (1 - DROP) * min(trace[:i]) for i in range(1, e))
    for stop in (0, e):
        tol, margin = tol_stopping_at(trace, stop)
        assert _by_hand_viol(trace, tol) == stop and margin >= MARGIN
        assert all(abs(v - tol) >= MARGIN * tol for v in trace[:stop + 1])
    tol, margin = tol_never(trace)
    assert _by_hand_viol(trace, tol) is None and margin >= 0.5
    assert replay_viol(trace, tol) == (len(trace) - 1, False)


def test_viol_choices_refuse_ties_and_zero():
    with pytest.raises(ValueError):
        first_drop([1.0, 1.0, 1.0 - 1e-9, 1.0])
    with pytest.raises(ValueError):
        tol_stopping_at([1.0, 1.0 - 1e-7, 0.5], 1)
    with pytest.raises(ValueError):
        tol_never([1.0, 0.0])


def _by_hand_plateau(trace, tol, n):
    count, best = 0, float("inf")
    for i, loss in enumerate(trace):
        count = count + 1 if loss > best - tol else 0
        best = min(best, loss)
        if count >= n:
            return i
    return None


# a loss trace that falls, rises once and falls again (the counter runs up and is reset), then flattens
PLATEAU = [0.70, 0.62, 0.60, 0.63, 0.55, 0.549, 0.5485, 0.5484, 0.5483, 0.5482]


@pytest.mark.parametrize("n_iter_no_change", [1, 2, 3])
def test_plateau_choice_stops_where_replayed(n_iter_no_change):
    tol, stop, margin, resets = choose_plateau_tol(PLATEAU, n_iter_no_change)
    assert _by_hand_plateau(PLATEAU, tol, n_iter_no_change) == stop < len(PLATEAU) - 1
    assert margin >= MARGIN
    crit = plateau_critical(PLATEAU)
    assert crit == [min(PLATEAU[:i]) - PLATEAU[i] for i in range(1, len(PLATEAU))]
    assert all(abs(tol - crit[i - 1]) >= MARGIN * PLATEAU[i] for i in range(1, stop + 1))
    assert replay_plateau(PLATEAU, tol, n_iter_no_change)[:2] == (stop, True)
    # the widest gap: no other adjacent pair of critical values that stops early (and resets, as this one does) is
    # wider
    assert resets > 0 or n_iter_no_change == 1
    c = sorted(set(crit))
    lo = max(x for x in c if x < tol)
    hi = min(x for x in c if x > tol)
    for a, b in zip(c[:-1], c[1:]):
        mid = 0.5 * (a + b)
        if _by_hand_plateau(PLATEAU, mid, n_iter_no_change) not in (None, len(PLATEAU) - 1) and \
                replay_plateau(PLATEAU, mid, n_iter_no_change)[2] >= (resets > 0):
            assert b - a <= hi - lo
    print("n_iter_no_change", n_iter_no_change, "tol", tol, "stop", stop, "margin", margin, "resets", resets)


def test_plateau_choice_refuses_ties():
    flat = [0.5, 0.5, 0.5, 0.5, 0.5, 0.5]
    with pytest.raises(ValueError):
        choose_plateau_tol(flat, 2)
    near = [0.5, 0.5 - 1e-9, 0.5 - 2e-9, 0.5 - 3e-9, 0.5 - 2.5e-9, 0.5 - 4e-9]
    with pytest.raises(ValueError):
        choose_plateau_tol(near, 1)


# ------------------------------------------------------------------------------ the oracle stops where replayed
def _small_problem(clf, seed=0):
    from sparsepoly_b200 import synth
    X = synth.uniform_sparse(400, 60, 8, seed)
    rng = np.random.RandomState(seed + 1)
    s = np.asarray(X @ rng.randn(60)).ravel() + 0.3 * rng.randn(400)
    return X, (np.where(s > np.median(s), 1.0, -1.0) if clf else s)


@pytest.mark.parametrize("solver,reg", [("pcd", "omegati"), ("pbcd", "omegacs"), ("pcd-all", "omegati"),
                                        ("pbcd-all", "l21")])
def test_oracle_viol_stop_bookkeeping(solver, reg):
    from oracle import oracle as O
    X, y = _small_problem(False)
    if solver.endswith("-all"):
        kw = dict(n_components=3, solver=solver[:-4], regularizer=reg, beta=0.1, gamma=1e-3, random_state=0)
        fit = lambda **k: O.fit_all_subsets(X, y, **kw, **k)      # noqa: E731
    else:
        kw = dict(degree=3, n_components=3, solver=solver, regularizer=reg, alpha=0.1, beta=0.1, gamma=1e-3,
                  random_state=0, fit_lower="explicit")
        fit = lambda **k: O.fit_fm(X, y, **kw, **k)               # noqa: E731
    E = 8
    ref = fit(max_iter=E, tol=-1.0)
    trace = ref["trace"]
    assert len(trace) == E and ref["n_iter_"] == E - 1 and not ref["converged"]
    e = first_drop(trace)
    for stop in sorted({0, e}):
        tol, margin = tol_stopping_at(trace, stop)
        out = fit(max_iter=E, tol=tol)
        assert out["n_iter_"] == stop and out["converged"], (stop, tol, out["n_iter_"])
        assert out["trace"] == trace[:stop + 1]
        print(solver, reg, "stop", stop, "tol", tol, "margin", margin)
    tol, _ = tol_never(trace)
    out = fit(max_iter=E, tol=tol)
    assert out["n_iter_"] == E - 1 and not out["converged"] and out["trace"] == trace


@pytest.mark.parametrize("n_iter_no_change", [1, 2, 3])
def test_oracle_plateau_stop_bookkeeping(n_iter_no_change):
    from oracle import oracle as O
    X, y = _small_problem(True)
    kw = dict(degree=2, loss="logistic", n_components=3, solver="psgd", regularizer="l1", alpha=1e-3, beta=1e-3,
              gamma=1e-3, eta0=20.0, learning_rate="constant", batch_size=50, shuffle=True, random_state=0)
    E = 12
    ref = O.fit_fm(X, y, max_iter=E, tol=-1.0, n_iter_no_change=10 ** 9, **kw)
    trace = ref["trace"]
    assert ref["n_iter_"] == E - 1 and not ref["converged"]
    tol, stop, margin, resets = choose_plateau_tol(trace, n_iter_no_change)
    out = O.fit_fm(X, y, max_iter=E, tol=tol, n_iter_no_change=n_iter_no_change, **kw)
    assert out["n_iter_"] == stop and out["converged"] and out["trace"] == trace[:stop + 1]
    assert min(plateau_critical(trace)) < 0.0                 # (the loss rises: the schedule is that aggressive)
    assert resets > 0 or n_iter_no_change == 1
    print("n_iter_no_change", n_iter_no_change, "tol", tol, "stop", stop, "margin", margin, "resets", resets)
