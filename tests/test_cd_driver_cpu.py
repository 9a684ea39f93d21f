"""The pcd / pbcd driver shared by fit and fit_many (sparsepoly_b200/cd.py), without a device: the stopping loop
driven by scripted violation sums and a fake epoch, and the sub-epoch order of every model shape."""
import itertools
import warnings

import pytest

import sparsepoly_b200 as S
from sparsepoly_b200 import cd
from test_stopping_cpu import parse_traces

NOT_CONVERGED = "Objective did not converge. Increase max_iter."


class Script:
    """A fake epoch over scripted violation sums: traces[i][it] is model i's sum at epoch it.  Records the active
    models of every epoch and, in `events`, every sync and callback in the order they happen."""

    def __init__(self, traces, capsys=None):
        self.traces, self.capsys = traces, capsys
        self.it, self.active, self.events, self.printed = 0, [], [], []

    def syncs(self):
        return [lambda i=i: self.events.append(("sync", i)) for i in range(len(self.traces))]

    def callback(self, i, result=None, stop_at=None):
        def cb(est):
            self.events.append(("callback", i, self.it - 1))
            return result if stop_at is None or self.it - 1 == stop_at else None
        return cb

    def __call__(self, active):
        if self.capsys is not None:                      # what was printed before this epoch ran
            self.printed.append(self.capsys.readouterr().out)
        self.active.append(list(active))
        self.it += 1
        return [self.traces[i][self.it - 1] for i in active]


def _est(**kw):
    kw.setdefault("max_iter", 10)
    return S.SparseFactorizationMachineRegressor(**kw)


def _run(ests, script, buffered=False):
    with warnings.catch_warnings(record=True) as caught:
        warnings.simplefilter("always")
        converged = cd.stopping_loop(ests, script.syncs(), script, buffered=buffered)
    return converged, [str(w.message) for w in caught]


def test_one_model_stops_below_tol():
    est = _est(tol=0.9)
    script = Script([[5.0, 3.0, 1.0, 0.5, 0.1]])
    converged, warned = _run([est], script)
    assert converged == [True] and est.n_iter_ == 3 and warned == []
    assert script.active == [[0]] * 4
    assert script.events == [("sync", 0)]                # no callback: synced once, at the end


def test_one_model_runs_to_max_iter():
    est = _est(tol=0.1, max_iter=3)
    script = Script([[5.0, 3.0, 1.0, 0.5]])
    converged, warned = _run([est], script)
    assert converged == [False] and est.n_iter_ == 2 and warned == [NOT_CONVERGED]
    assert script.active == [[0]] * 3


def test_models_stop_at_their_own_epochs():
    """Models that stop at epochs 0, 1 and 3 and one that never does; later epochs run the others only."""
    ests = [_est(tol=tol, max_iter=6) for tol in (1.0, 2.0, 0.5, 0.0)]
    traces = [[0.5] + [9.0] * 5, [3.0, 1.5] + [9.0] * 4, [4.0, 3.0, 2.0, 0.25, 9.0, 9.0], [1.0] * 6]
    script = Script(traces)
    converged, warned = _run(ests, script)
    assert converged == [True, True, True, False]
    assert [e.n_iter_ for e in ests] == [0, 1, 3, 5]
    assert script.active == [[0, 1, 2, 3], [1, 2, 3], [2, 3], [2, 3], [3], [3]]
    assert warned == [NOT_CONVERGED]                     # one warning per unconverged model
    assert script.events == [("sync", i) for i in range(4)]


def test_callback_stops_and_sees_a_synced_model():
    """A callback returning non-None stops its model (not converged); sync runs before every callback call and once
    at the end; the callback runs every n_calls epochs, from epoch 0."""
    script = Script([[9.0] * 8, [9.0] * 8])
    ests = [_est(tol=1.0, max_iter=8, n_calls=2), _est(tol=1.0, max_iter=8, n_calls=3)]
    ests[0].callback = script.callback(0, result="stop", stop_at=4)
    ests[1].callback = script.callback(1)
    converged, warned = _run(ests, script)
    assert converged == [False, False] and [e.n_iter_ for e in ests] == [4, 7]
    assert warned == [NOT_CONVERGED, NOT_CONVERGED]
    calls = [(i, it) for kind, i, *rest in script.events if kind == "callback" for it in rest]
    assert [it for i, it in calls if i == 0] == [0, 2, 4]
    assert [it for i, it in calls if i == 1] == [0, 3, 6]
    for j, ev in enumerate(script.events):
        if ev[0] == "callback":
            assert script.events[j - 1] == ("sync", ev[1])
    assert script.events[-2:] == [("sync", 0), ("sync", 1)]
    assert script.active[-1] == [1] and len(script.active) == 8


def test_max_iter_zero_next_to_a_running_model():
    ests = [_est(tol=1.0, max_iter=0), _est(tol=-1.0, max_iter=2)]
    script = Script([[], [5.0, 4.0]])
    converged, warned = _run(ests, script)
    assert script.active == [[1], [1]]
    assert converged == [False, False] and [e.n_iter_ for e in ests] == [0, 1]
    assert warned == [NOT_CONVERGED, NOT_CONVERGED]
    assert script.events == [("sync", 0), ("sync", 1)]
    assert _run([_est(max_iter=0)], Script([[]]))[0] == [False]


TRACES = [[0.30000000000000004, 1 / 3, 2.5e-17], [7.0, 6.5, 6.25, 6.125]]


def _verbose_ests():
    return [_est(tol=1e-16, max_iter=4, verbose=True), _est(tol=0.0, max_iter=4, verbose=True)]


def test_verbose_lines_print_as_the_epochs_run(capsys):
    """One model (a single fit): each epoch's line is printed before the next epoch runs."""
    script = Script(TRACES[:1], capsys)
    _run(_verbose_ests()[:1], script)
    out = capsys.readouterr().out
    assert script.printed == ["", "Iteration 1 violation sum 0.30000000000000004\n",
                              "Iteration 2 violation sum 0.3333333333333333\n"]
    assert out == "Iteration 3 violation sum 2.5e-17\nConverged at iteration 3\n"
    assert parse_traces("".join(script.printed) + out) == TRACES[:1]


def test_buffered_verbose_lines_come_model_by_model(capsys):
    """Many models (fit_many): nothing is printed while the epochs run, then each model's lines in list order, which
    carry its violation sums exactly."""
    script = Script(TRACES, capsys)
    _run(_verbose_ests(), script, buffered=True)
    out = capsys.readouterr().out
    assert script.printed == [""] * 4
    assert parse_traces(out) == TRACES
    assert out.index("Converged at iteration 3\n") < out.index("Iteration 1 violation sum 7.0\n")


FM_CASES = list(itertools.product(("pcd", "pbcd"), (2, 3, 4, 5), ("explicit", "augment", None), (True, False)))


@pytest.mark.parametrize("solver,degree,fit_lower,fit_linear", FM_CASES)
def test_fm_sub_epochs(solver, degree, fit_lower, fit_linear):
    """Linear CD, then the explicit lower orders ascending on P[degree - deg], then the top order on P[0]."""
    est = S.SparseFactorizationMachineRegressor(solver=solver, degree=degree, fit_lower=fit_lower,
                                                fit_linear=fit_linear)
    want = [("linear", None, None)] if fit_linear else []
    if fit_lower == "explicit":
        want += [(solver, deg, degree - deg) for deg in range(2, degree)]
    want.append((solver, degree, 0))
    assert cd.sub_epochs(est) == want


def test_fm_sub_epochs_spelled_out():
    est = S.SparseFactorizationMachineRegressor(solver="pcd", degree=4, fit_lower="explicit", fit_linear=True)
    assert cd.sub_epochs(est) == [("linear", None, None), ("pcd", 2, 2), ("pcd", 3, 1), ("pcd", 4, 0)]
    est = S.SparseFactorizationMachineRegressor(solver="pbcd", degree=3, fit_lower=None, fit_linear=False)
    assert cd.sub_epochs(est) == [("pbcd", 3, 0)]


@pytest.mark.parametrize("solver", ["pcd", "pbcd"])
def test_all_subsets_sub_epochs(solver):
    assert cd.sub_epochs(S.SparseAllSubsetsRegressor(solver=solver)) == [(solver, -1, 0)]
