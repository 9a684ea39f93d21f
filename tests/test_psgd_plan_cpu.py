"""CPU checks of the planned psgd path's host logic (sparsepoly_b200/psgd_plan.py) and of its algorithm:
the plan arrays the CUDA kernels read are replayed by a numpy model of those kernels
(tests/psgd_plan_model.py) and the result must equal the oracle's psgd fit (reference
optimizer/psgd.py:125-199) to 1e-9 -- single rank and sharded over 2 / 3 simulated ranks."""
import numpy as np
import pytest
import torch

import psgd_plan_model as M
from psgd_plan_model import RankState, run_model
from sparsepoly_b200 import synth
from sparsepoly_b200.distributed import interleave_shards
from sparsepoly_b200.psgd_plan import CHUNK, SHORT, PsgdPlan


def _csr_t(X):
    return (torch.from_numpy(X.indptr.astype(np.int32)), torch.from_numpy(X.indices.astype(np.int32)),
            torch.from_numpy(X.data.astype(np.float64)))


def _plans(Xs, idxs, d, b_loc, group_entries=48_000_000):
    G = len(Xs)
    plans = [PsgdPlan(_csr_t(X), torch.from_numpy(idx), d, b_loc, world=G, rank=r, group_entries=group_entries,
                      defer_owner_tables=G > 1) for r, (X, idx) in enumerate(zip(Xs, idxs))]
    if G > 1:
        lists = [p.column_lists() for p in plans]
        gathered = tuple([l[t] for l in lists] for t in range(4))
        for p in plans:
            p.finish_owner_tables(*gathered)
    return plans


@pytest.mark.parametrize("b_loc,group_entries", [(37, 48_000_000), (500, 900), (1, 48_000_000), (4000, 48_000_000)])
def test_plan_layout_matches_brute_force(b_loc, group_entries):
    X = synth.criteo_like(1500, 400, 3)                      # 13 dense columns: split over many chunks
    rng = np.random.RandomState(0)
    idx = rng.permutation(1500).astype(np.int32)
    plan = _plans([X], [idx], 400, b_loc, group_entries)[0]
    M = plan.n_minibatches
    assert M == -(-1500 // b_loc)
    e_pos, e_x = plan.e_pos.numpy(), plan.e_x.numpy()
    u_feat, u_ptr = plan.u_feat.numpy(), plan.u_ptr.numpy()
    for m in range(M):
        rows = idx[m * b_loc:(m + 1) * b_loc]
        want = []                                            # (feature, position, value) sorted by feature then position
        for pos, i in enumerate(rows):
            for e in range(X.indptr[i], X.indptr[i + 1]):
                want.append((int(X.indices[e]), pos, float(X.data[e])))
        want.sort(key=lambda t: (t[0], t[1]))
        e0, e1 = plan.mb_eptr[m], plan.mb_eptr[m + 1]
        assert e1 - e0 == len(want)
        u0, u1 = plan.mb_uptr[m], plan.mb_uptr[m + 1]
        got_feat = np.repeat(u_feat[u0:u1], np.diff(u_ptr[u0:u1 + 1]))
        assert np.array_equal(got_feat, [t[0] for t in want])
        assert np.array_equal(e_pos[e0:e1], [t[1] for t in want])
        assert np.array_equal(e_x[e0:e1], [t[2] for t in want])
        lens = np.diff(u_ptr[u0:u1 + 1])
        short = plan.sc_u.numpy()[plan.mb_shptr[m]:plan.mb_shptr[m + 1]]
        assert np.array_equal(short, u0 + np.nonzero((lens <= SHORT) & (lens > 1))[0])
        sc_ptr = plan.sc_ptr.numpy()[plan.mb_shptr[m]:plan.mb_shptr[m + 1] + 1]
        assert np.array_equal(np.diff(sc_ptr), lens[short - u0])
        sg = slice(plan.mb_sgptr[m], plan.mb_sgptr[m + 1])
        singles = u0 + np.nonzero(lens == 1)[0]
        assert np.array_equal(plan.sg_u.numpy()[sg], singles) and np.array_equal(plan.sg_feat.numpy()[sg], u_feat[singles])
        assert np.array_equal(plan.sg_pos.numpy()[sg], e_pos[u_ptr[singles]]) and np.array_equal(plan.sg_x.numpy()[sg], e_x[u_ptr[singles]])
        lc_u = plan.lc_u.numpy()[plan.mb_lcptr[m]:plan.mb_lcptr[m + 1]]
        lc_e0 = plan.lc_e0.numpy()[plan.mb_lcptr[m]:plan.mb_lcptr[m + 1]]
        want_u, want_e = [], []
        for u in u0 + np.nonzero(lens > SHORT)[0]:
            for e in range(u_ptr[u], u_ptr[u + 1], CHUNK):
                want_u.append(u); want_e.append(e)
        assert np.array_equal(lc_u, want_u) and np.array_equal(lc_e0, want_e)
        lsl = slice(plan.mb_lcptr[m], plan.mb_lcptr[m + 1])
        assert np.array_equal(plan.lc_feat.numpy()[lsl], u_feat[lc_u])
        want_cnt = [min(CHUNK, u_ptr[u + 1] - e) + ((1 << 30) if u_ptr[u + 1] - u_ptr[u] <= CHUNK else 0) for u, e in zip(want_u, want_e)]
        assert np.array_equal(plan.lc_cnt.numpy()[lsl], want_cnt)
        ml_u = plan.ml_u.numpy()[plan.mb_mlptr[m]:plan.mb_mlptr[m + 1]]
        ml_c0 = plan.ml_c0.numpy()[plan.mb_mlptr[m]:plan.mb_mlptr[m + 1]]
        assert np.array_equal(ml_u, u0 + np.nonzero(lens > CHUNK)[0])
        for u, c0 in zip(ml_u, ml_c0):
            assert lc_u[c0] == u and lc_e0[c0] == u_ptr[u] and (c0 == 0 or lc_u[c0 - 1] != u)
    assert plan.max_chunks == np.max(np.diff(plan.mb_lcptr)) and plan.max_cols == np.max(np.diff(plan.mb_uptr))


def _oracle_fit(X, y, kw, epochs):
    from oracle import oracle as O
    return O.fit_fm(X, y, max_iter=epochs, tol=-1.0, n_iter_no_change=10 ** 9, random_state=0, **kw)


CASES = [
    dict(degree=2, loss="logistic", n_components=5, solver="psgd", regularizer="squaredl12", alpha=1e-3, beta=1e-3,
         gamma=2e-3, eta0=0.2, fit_lower=None),
    dict(degree=3, loss="squared", n_components=3, solver="psgd", regularizer="l1", alpha=1e-2, beta=1e-2,
         gamma=1e-3, eta0=0.05, fit_lower="explicit", learning_rate="invscaling", power_t=0.5),
    dict(degree=2, loss="squared_hinge", n_components=4, solver="psgd", regularizer="squaredl12", alpha=1e-3,
         beta=1e-3, gamma=5e-3, eta0=0.1, fit_lower=None, fit_linear=False, learning_rate="constant"),
]


@pytest.mark.parametrize("world", [1, 2, 3])
@pytest.mark.parametrize("case", range(len(CASES)))
def test_plan_model_matches_oracle(case, world):
    kw = dict(CASES[case])
    n_loc, d, b_glob = 240, 90, 48 * world if world > 1 else 50
    if case == 2:
        b_glob = 240 * world                                   # one minibatch per epoch: the dense columns split
    Xs = [synth.criteo_like(n_loc, d, 11 + r) for r in range(world)]
    rng = np.random.RandomState(5)
    ys = [np.where(rng.rand(n_loc) < 0.4, 1.0, -1.0) if kw["loss"] != "squared" else rng.randn(n_loc) for _ in range(world)]
    idxs = [np.arange(n_loc, dtype=np.int32) for _ in range(world)]
    b_loc = max(1, b_glob // world)
    plans = _plans(Xs, idxs, d, b_loc)
    degree, k = kw["degree"], kw["n_components"]
    n_orders = degree - 1 if kw["fit_lower"] == "explicit" else 1
    ranks = [RankState(p, (X.indptr, X.indices, X.data), y, idx, n_orders, k, degree) for p, X, y, idx in zip(plans, Xs, ys, idxs)]
    P_kd = 0.01 * np.random.RandomState(0).randn(n_orders, k, d)              # what fit draws with random_state=0
    P = np.ascontiguousarray(P_kd.swapaxes(1, 2))
    w = np.zeros(d)
    epochs = 2
    it, sum_loss = run_model(ranks, d, n_orders, k, degree, kw["regularizer"], kw["loss"], kw.get("fit_linear", True),
                             np.ones(k), kw["alpha"], kw["beta"], kw["gamma"], kw["eta0"], kw.get("learning_rate", "optimal"),
                             kw.get("power_t", 1.0), 1, P, w, epochs=epochs)
    # the equivalent single-process run: shards interleaved in blocks of b_loc rows (distributed.interleave_shards)
    import scipy.sparse as sp
    order = interleave_shards([np.arange(n_loc) + r * n_loc for r in range(world)], b_loc * world)
    Xall, yall = sp.vstack(Xs).tocsr()[order], np.concatenate(ys)[order]
    out = _oracle_fit(Xall, yall, dict(kw, batch_size=b_loc * world), epochs)
    P_ref = out["P_"].swapaxes(1, 2)
    scale = np.max(np.abs(P_ref))
    assert np.max(np.abs(P - P_ref)) <= 1e-9 * scale
    assert np.max(np.abs(w - out["w_"])) <= 1e-9 * max(np.max(np.abs(out["w_"])), 1e-300)
    dust = (np.abs(P) < 1e-12 * scale) & (np.abs(P_ref) < 1e-12 * scale)
    assert np.all(((P != 0) == (P_ref != 0)) | dust)
    assert it == out["it_"]
    assert abs(sum_loss / (n_loc * world) - out["trace"][-1]) <= 1e-9 * abs(out["trace"][-1])
    assert 0.02 < np.mean(P_ref != 0) < 0.999 or kw["regularizer"] == "l1"


# ---------------------------------------------------------------- squared-l1,2 band solve (psgd_solve_kernel)
def _sorted_rule(vals, strength):
    """utils.py:26-70 restated with a sort: the largest theta with v_(theta) > 2 s S_theta / (1 + 2 s theta)."""
    v = np.sort(np.asarray(vals, dtype=np.float64))[::-1]
    cs = np.cumsum(v)
    tq = 2.0 * strength * cs / (1.0 + 2.0 * strength * np.arange(1, v.size + 1))
    ok = np.nonzero(v > tq)[0]
    m = int(ok.max()) + 1 if ok.size else 0
    return (2.0 * strength * cs[m - 1] / (1.0 + 2.0 * strength * m)) if m else 0.0, m


def test_band_exact_sum_is_order_independent_and_correctly_rounded():
    import math
    rng = np.random.RandomState(3)
    for trial in range(200):
        hi = 10.0 ** rng.uniform(-9, 3)
        E = int(np.floor(np.log2(hi))) + 1
        n = rng.randint(1, 2049)
        vals = hi * (1.0 - 0.18 * rng.rand(n))                       # inside (0.82 hi, hi]: the widest band (+-10 %)
        s0 = M.band_exact_sum(vals, E)
        assert s0 == M.band_exact_sum(vals[rng.permutation(n)], E)   # any order: the same bits
        assert s0 == math.fsum(vals)                                 # the exactly rounded sum


def test_band_solve_matches_the_sorted_rule():
    rng = np.random.RandomState(4)
    hits = 0
    for trial in range(400):
        n_all = rng.randint(5, 400)
        strength = 10.0 ** rng.uniform(-3, 1)
        vals = np.abs(rng.randn(n_all)) * 10.0 ** rng.uniform(-4, 1)
        tau_ref, theta = _sorted_rule(vals, strength)
        delta = rng.choice([0.002, 0.01, 0.02, 0.1])
        tp = tau_ref * (1.0 + 0.6 * delta * (2.0 * rng.rand() - 1.0))  # a prediction a little off the true threshold
        b_lo, b_hi = tp * (1.0 - delta), tp * (1.0 + delta)
        above = vals[vals > b_hi]
        band = vals[(vals > b_lo) & ~(vals > b_hi)]
        tau = M.band_solve(band[rng.permutation(band.size)], float(np.sum(above)), float(above.size), strength, b_lo, b_hi)
        assert tau is not None                                        # the true threshold is inside the band
        assert abs(tau - tau_ref) <= 1e-13 * tau_ref
        assert int(np.sum(vals > tau)) == theta
        hits += 1
    assert hits == 400


def test_band_solve_reports_a_miss():
    vals = np.array([1.0, 0.9, 0.8, 0.05, 0.04])
    strength = 0.3
    tau_ref, _ = _sorted_rule(vals, strength)
    for tp in (tau_ref * 1.5, tau_ref * 0.6):                          # prediction far off: the band does not hold tau
        b_lo, b_hi = tp * 0.98, tp * 1.02
        above = vals[vals > b_hi]
        band = vals[(vals > b_lo) & ~(vals > b_hi)]
        assert M.band_solve(band, float(above.sum()), float(above.size), strength, b_lo, b_hi) is None


# ---------------------------------------------------------------- long horizons of the lazy frame
def test_plan_model_folds_the_frame_inside_an_epoch():
    """batch_size=1 with eta * alpha = 0.5: Cw grows by 1.5 per minibatch and would overflow after ~1750 of them
    (every w then reads back as 0; w itself stays O(1), held by the loss).  The model folds the frame after every
    minibatch that takes Cw past 1e100 -- here three times inside one epoch -- and ends at the oracle's model."""
    n, d, k = 2000, 40, 4
    X = synth.uniform_sparse(n, d, 5, 11)
    y = np.where(np.random.RandomState(5).rand(n) < 0.4, 1.0, -1.0)
    kw = dict(degree=2, loss="logistic", n_components=k, solver="psgd", regularizer="squaredl12", alpha=1.0, beta=0.02,
              gamma=1e-4, eta0=0.5, learning_rate="constant", fit_lower=None)
    idx = np.arange(n, dtype=np.int32)
    plan = _plans([X], [idx], d, 1)[0]
    ranks = [RankState(plan, (X.indptr, X.indices, X.data), y, idx, 1, k, 2)]
    P = np.ascontiguousarray((0.01 * np.random.RandomState(0).randn(1, k, d)).swapaxes(1, 2))
    w = np.zeros(d)
    folds = []
    it, _ = run_model(ranks, d, 1, k, 2, "squaredl12", "logistic", True, np.ones(k), kw["alpha"], kw["beta"],
                      kw["gamma"], kw["eta0"], "constant", 1.0, 1, P, w, folds=folds)
    # Cw after the minibatch of `it` = 1.5 ** (minibatches since the last fold): folded after 568, 1136, 1704;
    # C = 1.01 ** 2000 stays far below the bound
    assert 1.5 ** 567 < 1e100 < 1.5 ** 568 and 1.01 ** n < 1e10
    assert folds == [568, 1136, 1704]
    out = _oracle_fit(X, y, dict(kw, batch_size=1), 1)
    P_ref = out["P_"].swapaxes(1, 2)
    assert 0.2 < np.mean(P_ref != 0) and np.all(np.isfinite(P)) and np.max(np.abs(out["w_"])) > 1e-3
    assert np.max(np.abs(P - P_ref)) <= 1e-9 * np.max(np.abs(P_ref))
    assert np.array_equal(P != 0, P_ref != 0)
    assert np.max(np.abs(w - out["w_"])) <= 1e-9 * np.max(np.abs(out["w_"]))
    assert it == out["it_"] == n + 1
