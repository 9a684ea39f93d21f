"""The window sweeps (wplan.cu, pcd_window.cu, pbcd_window.cu) at the limits of their engine CTA's fixed tables,
against the host restatement of tests/wplan_model.py and against the C oracle:
  * the plan arrays (cflag hot bits, ht_ptr, ht_cls, n_slots, slot rows, the packed hot nonzeros) bit for bit;
  * windows with exactly slot_cap slots (pcd record strides 4 and 8, pbcd at k = 32), a position with exactly 32
    chain-warp nonzeros, pcd windows of 128 / 129 / 192 / 256 positions around the 128-position speculation mask,
    pbcd windows of 33..64 positions, last windows of one position, d < B, d == B, a window without hot nonzeros
    and a sample touched by every position of a window;
  * one step past each limit: cap + 1 slots, 33 chain nonzeros, windows above 256 (pcd) / 64 (pbcd).
Every fit asserts that its plan reached the limit it names (plan mode and stats, speculation counters), so a plan
that silently fell back fails, and is also compared with the cluster sweep on the same input."""
import numpy as np
import pytest
import scipy.sparse as sp

import wplan_model as M
from golden_util import rel_err, same_support
from test_parity_gpu import _check_objective, _fit, _wspec_read

pytestmark = pytest.mark.gpu

TOL = 1e-9
ERRORS = {}


def _lib():
    from sparsepoly_b200 import _lib as L
    return L.load()


def _background(n, d, r, seed):
    from sparsepoly_b200 import synth
    return synth.uniform_sparse(n, d, r, seed)


def _singles(n, d, seed):
    """n samples of one nonzero each: cold at any window size."""
    rng = np.random.RandomState(seed)
    X = sp.csr_matrix((rng.randn(n), rng.randint(0, d, n), np.arange(n + 1)), shape=(n, d))
    X.sort_indices()
    return X


def _targets(X, seed, degree, clf):
    from sparsepoly_b200 import synth
    from oracle import oracle as O
    Pt = synth.planted_P(X.shape[1], 3, seed + 1, frac_features=0.3, scale=0.5)
    s = O.poly_predict(X, Pt, np.ones(3), "anova", max(degree, 2)) if degree != -1 else \
        O.poly_predict(X, 0.3 * Pt, np.ones(3), "all-subsets")
    return synth.targets_from_scores(s, seed + 2, clf)


def _estimator(kw, all_subsets=False):
    import sparsepoly_b200 as S
    clf = kw.get("loss", "squared") != "squared"
    ekw = dict(kw)
    if not clf:
        ekw.pop("loss", None)
    if all_subsets:
        return (S.SparseAllSubsetsClassifier if clf else S.SparseAllSubsetsRegressor)(**ekw)
    return (S.SparseFactorizationMachineClassifier if clf else S.SparseFactorizationMachineRegressor)(**ekw)


_ORACLE = {}


def _oracle(key, X, y, kw, all_subsets=False):
    from oracle import oracle as O
    if key not in _ORACLE:
        okw = dict(kw)
        okw.setdefault("loss", "squared")
        _ORACLE[key] = O.fit_all_subsets(X, y, **okw) if all_subsets else O.fit_fm(X, y, **okw)
    return _ORACLE[key]


def _run(tag, key, X, y, kw, monkeypatch, env, all_subsets=False):
    """Window fit with `env`, checked against the oracle; then the cluster sweep on the same input.
    Returns (est, oracle output, speculation counters)."""
    out = _oracle(key, X, y, kw, all_subsets)
    for k in ("SPARSEPOLY_B200_WINDOW", "SPARSEPOLY_B200_HORIZON", "SPARSEPOLY_B200_NEAR"):
        monkeypatch.delenv(k, raising=False)
    monkeypatch.setenv("SPARSEPOLY_B200_SWEEP", "window")
    for k, v in env.items():
        monkeypatch.setenv(k, str(v))
    _wspec_read()
    est = _fit(_estimator(kw, all_subsets), X, y)
    spec = _wspec_read()
    err = rel_err(est.P_, out["P_"])
    assert err <= TOL, (tag, err)
    assert same_support(est.P_, out["P_"]), tag
    if "w_" in out and hasattr(est, "w_"):
        assert rel_err(est.w_, out["w_"]) <= TOL, tag
    assert est.n_iter_ == out["n_iter_"], tag
    _check_objective(est, X, y, out["P_"], out.get("w_"))
    monkeypatch.setenv("SPARSEPOLY_B200_SWEEP", "cluster")
    estc = _fit(_estimator(kw, all_subsets), X, y)
    assert estc._dev_state["plan"].mode == "cluster"
    errc = rel_err(est.P_, estc.P_)
    assert errc <= TOL and np.array_equal(est.P_ != 0, estc.P_ != 0), (tag, errc)
    ERRORS[tag] = (err, errc)
    return est, out, spec


def _report(tag, plan, cap, spec, extra=""):
    st = plan.wplan.stats
    err, errc = ERRORS[tag]
    print(f"{tag}: window {st['window']} horizon {st['horizon']} near {st['near']} max_slots {st['max_slots']} / "
          f"slot_cap {cap}, speculated {spec[0]} rejected {spec[1]}, rel err vs oracle {err:.2e}, "
          f"vs cluster sweep {errc:.2e} {extra}")


# ===================================================================================== plan vs restatement
def _check_plan(X, B, H, near, pbcd_shape=None):
    """WindowPlan (identity order) against wplan_model, array by array; a forced window that does not fit must
    raise exactly when the restatement overflows at near and at 0."""
    import torch
    from sparsepoly_b200.dataset import DeviceDataset, WindowPlan
    ds = DeviceDataset(X, need_csr=True, need_csc=True)
    wp = WindowPlan(ds, 4, window=B, horizon=H, pbcd_shape=pbcd_shape)
    if pbcd_shape is None:
        wp.near = near
        cap, ent = M.pcd_slot_cap(4), M.PCD_ENT_PER_SLOT
    else:
        near = 0
        cap, ent = M.pbcd_slot_cap(*pbcd_shape), M.PBCD_ENT_PER_SLOT
    assert wp.slot_cap == cap
    d = X.shape[1]
    want_near = M.built_near(X, B, H, near, cap, ent)
    idx = torch.arange(d, dtype=torch.int32, device=ds.device)
    if want_near is None:
        with pytest.raises(ValueError, match="does not fit"):
            wp.build(idx)
        return None
    assert wp.build(idx)
    p = M.window_plan(X, B, H, want_near, cap, ent)
    st = wp.stats
    assert (st["window"], st["horizon"], st["near"], st["max_slots"]) == (B, H, want_near, p.max_slots), st
    cflag = wp.cflag[:ds.nnz].cpu().numpy()
    Xc = sp.csc_matrix(X)
    Xc.sort_indices()
    assert np.array_equal(cflag < 0, p.hot)
    assert np.array_equal(cflag & 0x7fffffff, Xc.indices)
    ht_ptr = wp.ht_ptr.cpu().numpy().astype(np.int64)
    assert np.array_equal(np.diff(ht_ptr), p.hot_count)
    assert np.array_equal(wp.n_slots.cpu().numpy(), p.n_slots)
    assert np.array_equal(wp.ht_cls[:d].cpu().numpy(), p.ht_cls)
    slot_row = wp.slot_row.cpu().numpy().reshape(-1, cap)
    h_sd = wp.h_sd.cpu().numpy().astype(np.int64)
    h_x = wp.h_x.cpu().numpy()
    for w in range(p.n_windows):
        rows = slot_row[w, :p.n_slots[w]]
        assert np.array_equal(np.sort(rows), p.slots[w]), w
        for t in range(w * B, min(d, (w + 1) * B)):
            got = [(int(rows[s & 0xffff]), ((s >> 16) & 0x1ff) - 1, bool(s & 0x40000000), bool(s & 0x20000000),
                    float(x)) for s, x in zip(h_sd[ht_ptr[t]:ht_ptr[t + 1]], h_x[ht_ptr[t]:ht_ptr[t + 1]])]
            assert got == p.ent[t], t
    return p


def _plan_inputs():
    cap = M.pcd_slot_cap(4)
    bg = _background(6000, 1920, 4, 21)
    return {
        "slot_cap": M.with_slots(bg, 96, 0, 4, cap, 1, cap),
        "chain32": M.with_chain(bg, 96 * 5 + 40, 11, 10, 11, 1, 2),
        "chain33": M.with_chain(bg, 96 * 5 + 40, 17, 0, 16, 2, 2),
        "full_chain": M.with_full_chain(bg, 3, 96, 3),
        "no_hot": M.without_hot(bg, 96, 1, 4),
    }


@pytest.mark.parametrize("B", [1, 7, 96, 128, 129, 256])
@pytest.mark.parametrize("off", [0, 1, -1])
def test_plan_matches_restatement_random(B, off):
    """Random inputs with d = 0, 1, B - 1 (mod B): the last window full, of one position, one short."""
    if B == 1 and off != 0:
        pytest.skip("every d is a multiple of 1")
    m = max(2, 600 // B)
    d = B * m + (off if off >= 0 else B - 1) if B > 1 else 400
    X = _background(2000, d, 4, B + 3 * (off + 1))
    for H in (0, 1):
        for near in (0, 1, 2):
            _check_plan(X, B, H, near)


@pytest.mark.parametrize("name", ["slot_cap", "chain32", "chain33", "full_chain", "no_hot"])
def test_plan_matches_restatement_at_limits(name):
    X = _plan_inputs()[name]
    for B in (96, 128, 256):
        for H in (0, 1):
            for near in (0, 1, 2):
                p = _check_plan(X, B, H, near)
                if (name, B, H) == ("slot_cap", 96, 0):
                    assert p.max_slots == M.pcd_slot_cap(4) and p.n_ent.max() == p.ent_cap
                if (name, B, near) == ("chain32", 96, 1):
                    assert p.chain.max() == 32
                if (name, B, near) == ("chain33", 96, 2):
                    assert p is None or p.near == 0


@pytest.mark.parametrize("k", [8, 32])
@pytest.mark.parametrize("B", [1, 7, 48, 64])
def test_pbcd_plan_matches_restatement(k, B):
    cap = M.pbcd_slot_cap(2, k)
    assert int(_lib().sp_pbcd_wplan_slot_cap(2, k)) == cap
    bg = _background(3000, 960, 3, 31)
    for X in (bg, M.with_slots(bg, 48, 1, 5, cap, 4, cap, M.PBCD_ENT_PER_SLOT)):
        for H in (0, 1):
            _check_plan(X, B, H, 0, pbcd_shape=(2, k))


def test_slot_caps_match_library():
    lib = _lib()
    for stride in (2, 4, 8):
        assert int(lib.sp_wplan_slot_cap(stride)) == M.pcd_slot_cap(stride)
    for deg in (2, 3, 4, 5, -1):
        for k in (1, 8, 31, 32, 33):
            assert int(lib.sp_pbcd_wplan_slot_cap(deg, k)) == M.pbcd_slot_cap(deg, k)


# ===================================================================================== fits at the limits
def _fm_kw(degree, loss, reg, **extra):
    kw = dict(degree=degree, loss=loss, n_components=4, solver="pcd", regularizer=reg, alpha=1e-4, beta=1e-5,
              gamma=1e-6, max_iter=2, tol=-1.0, random_state=0, mean=True, fit_lower="explicit")
    kw.update(extra)
    return kw


PCD_SLOT_CASES = [
    # (tag, degree (-1: all-subsets), loss, regularizer, horizon)
    ("fm3_l1_squared_h0", 3, "squared", "l1", 0),
    ("fm3_omegati_logistic_h1", 3, "logistic", "omegati", 1),
    ("fm4_omegati_squared_h0", 4, "squared", "omegati", 0),
    ("fm4_l1_logistic_h1", 4, "logistic", "l1", 1),
    ("all_omegati_squared_h1", -1, "squared", "omegati", 1),
]


@pytest.mark.parametrize("tag,degree,loss,reg,H", PCD_SLOT_CASES, ids=[c[0] for c in PCD_SLOT_CASES])
def test_pcd_window_at_slot_cap(tag, degree, loss, reg, H, monkeypatch):
    """One window of 96 positions with exactly slot_cap hot samples (record stride 4 at degree <= 3 and
    all-subsets, 8 at degree 4).  With fit_linear the linear sub-epoch runs on the same plan."""
    from sparsepoly_b200 import solvers
    stride = solvers.rec_stride(degree)
    cap = M.pcd_slot_cap(stride)
    B, w = 96, 7
    X = M.with_slots(_background(10000, 1920, 4, 40 + H), B, H, w, cap, 5, cap)
    y = _targets(X, 50, degree, loss != "squared")
    if degree == -1:
        kw = dict(loss=loss, n_components=4, solver="pcd", regularizer=reg, beta=1e-4, gamma=1e-5, mean=True,
                  max_iter=2, tol=-1.0, random_state=0)
    else:
        kw = _fm_kw(degree, loss, reg)
    near = M.built_near(X, B, H, 1, cap)
    assert near is not None
    est, out, spec = _run(tag, tag, X, y, kw, monkeypatch, {"SPARSEPOLY_B200_WINDOW": B, "SPARSEPOLY_B200_HORIZON": H},
                          all_subsets=degree == -1)
    plan = est._dev_state["plan"]
    assert plan.mode == "window", plan.mode
    st = plan.wplan.stats
    assert plan.wplan.slot_cap == cap == int(_lib().sp_wplan_slot_cap(stride))
    assert (st["window"], st["horizon"], st["near"], st["max_slots"]) == (B, H, near, cap), st
    assert int(plan.wplan.n_slots[w].item()) == cap
    _report(tag, plan, cap, spec)


PBCD_SLOT_CASES = [(deg, reg, H) for deg in (2, 3) for reg in ("l21", "omegacs") for H in (0, 1)]


@pytest.mark.parametrize("degree,reg,H", PBCD_SLOT_CASES)
def test_pbcd_window_at_slot_cap(degree, reg, H, monkeypatch):
    """pbcd at k = 32: one window of 48 positions with exactly sp_pbcd_wplan_slot_cap(degree, 32) slots.  The
    linear sub-epoch (fit_linear) has its own pcd plan of record stride 2 at the same window, below its cap."""
    cap = M.pbcd_slot_cap(degree, 32)
    B, w = 48, 11
    X = M.with_slots(_background(8000, 1920, 3, 60 + H), B, H, w, cap, 6, cap, M.PBCD_ENT_PER_SLOT)
    y = _targets(X, 70, degree, False)
    kw = dict(degree=degree, n_components=32, solver="pbcd", regularizer=reg, alpha=1e-4, beta=1e-4,
              gamma={"l21": 1e-4, "omegacs": 1e-6}[reg], max_iter=2, tol=-1.0, random_state=0, mean=True)
    tag = f"pbcd_deg{degree}_{reg}_h{H}"
    est, out, spec = _run(tag, tag, X, y, kw, monkeypatch, {"SPARSEPOLY_B200_WINDOW": B, "SPARSEPOLY_B200_HORIZON": H})
    plan, plan_lin = est._dev_state["plan"], est._dev_state["plan_lin"]
    assert plan.mode == "window" and plan_lin.mode == "window", (plan.mode, plan_lin.mode)
    st = plan.wplan.stats
    assert (st["window"], st["horizon"], st["near"], st["max_slots"]) == (B, H, 0, cap), st
    lin = plan_lin.wplan.stats
    assert plan_lin.wplan.slot_cap == M.pcd_slot_cap(2)
    assert lin["window"] == B and lin["max_slots"] == M.window_plan(X, B, H, 0, 1 << 30).max_slots < M.pcd_slot_cap(2)
    _report(tag, plan, cap, spec, f"(linear plan: max_slots {lin['max_slots']} / {plan_lin.wplan.slot_cap})")


@pytest.mark.parametrize("B", [33, 64])
def test_pbcd_wide_windows(B, monkeypatch):
    """pbcd windows of 33 and 64 positions (BWIN = 64), d = 1 (mod B) at 64."""
    d = 1921 if B == 64 else 1920
    X = _background(8000, d, 3, 80)
    y = _targets(X, 81, 2, False)
    kw = dict(degree=2, n_components=32, solver="pbcd", regularizer="omegacs", alpha=1e-4, beta=1e-4, gamma=1e-6,
              max_iter=2, tol=-1.0, random_state=0, mean=True)
    tag = f"pbcd_window{B}"
    est, out, spec = _run(tag, tag, X, y, kw, monkeypatch, {"SPARSEPOLY_B200_WINDOW": B, "SPARSEPOLY_B200_HORIZON": 1})
    plan = est._dev_state["plan"]
    assert plan.mode == "window" and plan.wplan.stats["window"] == B
    assert plan.wplan.stats["max_slots"] == M.window_plan(X, B, 1, 0, 1 << 30, order=None).max_slots
    _report(tag, plan, plan.wplan.slot_cap, spec)


@pytest.mark.parametrize("near", [1, 2])
@pytest.mark.parametrize("n_late,n_both,n_fwd", [(16, 0, 16), (11, 10, 11), (17, 0, 16)])
def test_chain_warp_lanes(n_late, n_both, n_fwd, near, monkeypatch):
    """A position handing exactly 32 nonzeros to the chain warp (late only + fwd only, or all three classes); 33
    overflows and the plan is rebuilt with near = 0."""
    lanes = n_late + n_both + n_fwd
    B, t = 96, 96 * 5 + 40
    X = M.with_chain(_background(10000, 1920, 4, 90), t, n_late, n_both, n_fwd, near, 7)
    y = _targets(X, 91, 3, True)
    kw = _fm_kw(3, "logistic", "omegati")
    tag = f"chain_{n_late}_{n_both}_{n_fwd}_near{near}"
    est, out, spec = _run(tag, ("chain", n_late, n_both, n_fwd, near), X, y, kw, monkeypatch,
                          {"SPARSEPOLY_B200_WINDOW": B, "SPARSEPOLY_B200_HORIZON": 0, "SPARSEPOLY_B200_NEAR": near})
    plan = est._dev_state["plan"]
    assert plan.mode == "window"
    want_near = near if lanes <= 32 else 0
    assert plan.wplan.stats["near"] == want_near, plan.wplan.stats
    cls = int(plan.wplan.ht_cls[t].item())
    if lanes <= 32:
        assert cls == n_late | (n_both << 8) | (n_fwd << 16)
    else:
        assert cls == 0
    _report(tag, plan, plan.wplan.slot_cap, spec, f"(chain lanes at position {t}: {lanes})")


SPEC_KW = dict(degree=2, n_components=4, solver="pcd", regularizer="squaredl12", beta=1e-5, gamma=1e-6, alpha=1e-3,
               max_iter=3, tol=-1.0, random_state=0, mean=True)


@pytest.mark.parametrize("B,d", [(128, 1920), (129, 1935), (192, 1920), (256, 1792), (192, 1828), (256, 1636)])
def test_speculation_window_widths(B, d, monkeypatch):
    """KIND_FM speculates only in windows of at most 128 positions (128-bit mover masks).  Full windows of
    129..256 positions never speculate; with a partial last window of 100 positions only that window may."""
    X = _background(10000, d, 5, 11)
    y = _targets(X, 12, 2, False)
    tag = f"spec_B{B}_d{d}"
    est, out, spec = _run(tag, ("spec", d), X, y, SPEC_KW, monkeypatch, {"SPARSEPOLY_B200_WINDOW": B})
    plan = est._dev_state["plan"]
    assert plan.mode == "window" and plan.wplan.stats["window"] == B
    frac = float(np.mean(out["P_"] != 0))
    assert 0.0 < frac < 0.3, frac
    nb_last = d - (d - 1) // B * B
    if B <= M.SPEC_WINDOW_MAX:
        assert spec[0] > 0, "speculation never engaged"
    elif nb_last > M.SPEC_WINDOW_MAX:
        assert spec == (0, 0), spec
    else:
        # each sweep of the last window commits at most nb_last speculative positions and counts each of at most
        # 4 rejections once more
        sweeps = SPEC_KW["n_components"] * SPEC_KW["max_iter"]
        assert 0 < spec[0] <= (nb_last + 4) * sweeps, spec
    _report(tag, plan, plan.wplan.slot_cap, spec, f"(last window {nb_last} positions, nonzero fraction {frac:.3f})")


EDGE_KW = _fm_kw(3, "logistic", "omegati")


def _edge_input(name):
    bg = _background(10000, 1920, 4, 100)
    if name == "d_1_mod_B":
        return _background(10000, 1921, 4, 100), 96, 1
    if name == "no_hot":
        return M.without_hot(bg, 96, 1, 6), 96, 1
    if name == "full_chain":
        return M.with_full_chain(bg, 6, 96, 8), 96, 0
    if name == "d_lt_B":
        return M.with_slots(_singles(6000, 200, 9), 256, 0, 0, 2000, 10, M.pcd_slot_cap(4)), 256, 0
    if name == "d_eq_B":
        return M.with_slots(_singles(6000, 256, 9), 256, 1, 0, M.pcd_slot_cap(4), 10, M.pcd_slot_cap(4)), 256, 1
    raise KeyError(name)


@pytest.mark.parametrize("name", ["d_1_mod_B", "no_hot", "full_chain", "d_lt_B", "d_eq_B"])
def test_window_edges(name, monkeypatch):
    """Last window of one position with horizon 1 (no next window), a window with no hot nonzero, one sample at
    every position of a window, d < B and d == B (one window; d == B at slot_cap)."""
    X, B, H = _edge_input(name)
    d = X.shape[1]
    kw = EDGE_KW if d > B else dict(SPEC_KW, max_iter=2)       # (rows of <= 2 nonzeros: degree 2)
    y = _targets(X, 101, kw["degree"], kw.get("loss", "squared") != "squared")
    est, out, spec = _run(name, name, X, y, kw, monkeypatch, {"SPARSEPOLY_B200_WINDOW": B, "SPARSEPOLY_B200_HORIZON": H})
    plan = est._dev_state["plan"]
    assert plan.mode == "window"
    p = M.window_plan(X, B, H, plan.wplan.stats["near"], M.pcd_slot_cap(4))
    assert plan.wplan.stats["window"] == B and plan.wplan.stats["max_slots"] == p.max_slots
    assert np.array_equal(plan.wplan.n_slots.cpu().numpy(), p.n_slots)
    if name == "no_hot":
        assert p.n_slots[6] == 0
    if name == "d_eq_B":
        assert p.max_slots == M.pcd_slot_cap(4)
    _report(name, plan, plan.wplan.slot_cap, spec)


def test_shuffled_single_window_at_slot_cap(monkeypatch):
    """shuffle=True with d == B: the plan is rebuilt every epoch, and every order of one window has the same
    slot set, here exactly slot_cap."""
    cap = M.pcd_slot_cap(4)
    X = M.with_slots(_singles(6000, 256, 9), 256, 0, 0, cap, 10, cap)
    y = _targets(X, 111, 2, False)
    kw = dict(SPEC_KW, max_iter=2, shuffle=True)
    est, out, spec = _run("shuffle_d_eq_B", "shuffle_d_eq_B", X, y, kw, monkeypatch, {"SPARSEPOLY_B200_WINDOW": 256})
    plan = est._dev_state["plan"]
    assert plan.mode == "window" and plan.wplan.stats["max_slots"] == cap
    assert not np.array_equal(plan._order_host, np.arange(256))          # the last plan is of a shuffled order
    _report("shuffle_d_eq_B", plan, cap, spec)


# ===================================================================================== one step past each limit
def _valid_fit_after():
    """A valid window fit in the same process still matches the oracle."""
    from oracle import oracle as O
    X = _background(20000, 1000, 5, 120)
    y = _targets(X, 121, 2, False)
    est = _fit(_estimator(SPEC_KW), X, y)
    assert est._dev_state["plan"].mode == "window"
    out = O.fit_fm(X, y, loss="squared", **SPEC_KW)
    assert rel_err(est.P_, out["P_"]) <= TOL and same_support(est.P_, out["P_"])


def test_forced_window_over_slot_cap_raises(monkeypatch):
    cap = M.pcd_slot_cap(4)
    X = M.with_slots(_background(10000, 1920, 4, 40), 96, 0, 7, cap + 1, 5, cap)
    assert M.built_near(X, 96, 0, 1, cap) is None
    y = _targets(X, 50, 3, False)
    monkeypatch.setenv("SPARSEPOLY_B200_SWEEP", "window")
    monkeypatch.setenv("SPARSEPOLY_B200_WINDOW", "96")
    with pytest.raises(ValueError, match=f"needs {cap + 1} slots"):
        _fit(_estimator(_fm_kw(3, "squared", "l1")), X, y)
    monkeypatch.delenv("SPARSEPOLY_B200_WINDOW")
    _valid_fit_after()


def test_auto_window_over_slot_cap_falls_back(monkeypatch):
    """auto: 96 positions would need cap + 1 slots, so the plan takes the next window size that fits (per the
    restatement), or the cluster sweep when none does."""
    cap = M.pcd_slot_cap(4)
    X = M.with_slots(_background(10000, 1920, 4, 40), 96, 0, 7, cap + 1, 5, cap)
    y = _targets(X, 50, 3, False)
    monkeypatch.setenv("SPARSEPOLY_B200_SWEEP", "auto")
    monkeypatch.setenv("SPARSEPOLY_B200_HORIZON", "0")
    kw = _fm_kw(3, "squared", "l1")
    est = _fit(_estimator(kw), X, y)
    plan = est._dev_state["plan"]
    cands = plan.wplan._candidates()
    assert 96 in cands
    expect = None
    for B in cands:
        p = M.window_plan(X, B, 0, 0, cap)
        if p.hot.sum() <= 0.5 * X.nnz and M.built_near(X, B, 0, 1, cap) is not None:
            expect = B
            break
    assert expect != 96
    if expect is None:
        assert plan.mode == "cluster"
    else:
        assert plan.mode == "window" and plan.wplan.stats["window"] == expect, plan.wplan.stats
    print("auto with", cap + 1, "slots at 96:", plan.mode, plan.wplan.stats if plan.mode == "window" else "")
    out = _oracle("auto_cap1", X, y, kw)
    assert rel_err(est.P_, out["P_"]) <= TOL and same_support(est.P_, out["P_"])


@pytest.mark.parametrize("solver,B", [("pcd", 257), ("pbcd", 65), ("pcd", 0)])
def test_window_above_engine_tables_raises(solver, B, monkeypatch):
    """A forced window above the engine's per-position tables (256 pcd, 64 pbcd) is a ValueError of the plan,
    raised before any launch."""
    X = _background(5000, 600, 4, 130)
    y = _targets(X, 131, 2, False)
    monkeypatch.setenv("SPARSEPOLY_B200_SWEEP", "window")
    monkeypatch.setenv("SPARSEPOLY_B200_WINDOW", str(B))
    kw = dict(SPEC_KW, solver=solver, max_iter=1, regularizer="omegacs" if solver == "pbcd" else "omegati")
    wmax = 256 if solver == "pcd" else 64
    with pytest.raises(ValueError, match=f"window={B} is outside 1..{wmax}"):
        _fit(_estimator(kw), X, y)
    monkeypatch.delenv("SPARSEPOLY_B200_WINDOW")
    _valid_fit_after()
