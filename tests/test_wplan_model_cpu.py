"""The window-plan restatement of tests/wplan_model.py against a brute-force statement of the same rule, and every
input constructor against the limit it is meant to hit."""
import numpy as np
import pytest
import scipy.sparse as sp

import wplan_model as M


def _brute(X, order, B, H, near):
    """Hot bits, slots and chain classes by direct search: for every hot nonzero look at every other nonzero of
    its sample, and for every position walk back through the window."""
    X = sp.csr_matrix(X)
    Xc = sp.csc_matrix(X)
    Xc.sort_indices()
    d = X.shape[1]
    pos = {int(j): t for t, j in enumerate(order)}
    row_cols = [set(X.indices[X.indptr[i]:X.indptr[i + 1]].tolist()) for i in range(X.shape[0])]
    hot = []
    touched = {}                                   # position -> hot samples
    for j in range(d):
        for e in range(Xc.indptr[j], Xc.indptr[j + 1]):
            i = int(Xc.indices[e])
            h = any(abs(pos[c] // B - pos[j] // B) <= H for c in row_cols[i] if c != j)
            hot.append(h)
            if h:
                touched.setdefault(pos[j], []).append(i)
    n_windows = (d + B - 1) // B
    slots = [sorted({i for t in range(w * B, min(d, (w + 1) * B)) for i in touched.get(t, [])})
             for w in range(n_windows)]
    ht_cls = np.zeros(d, dtype=np.int64)
    for t in range(d):
        w0 = (t // B) * B
        late = fwd = both = 0
        for i in touched.get(t, []):
            prev = [u for u in range(w0, t) if i in touched.get(u, [])]
            nxt = [u for u in range(t + 1, min(d, w0 + B)) if i in touched.get(u, [])]
            is_late = bool(prev) and t - prev[-1] <= near
            is_fwd = bool(nxt) and nxt[0] - t <= near
            late += is_late and not is_fwd
            both += is_late and is_fwd
            fwd += is_fwd and not is_late
        ht_cls[t] = late | (both << 8) | (fwd << 16)
    return np.array(hot), slots, ht_cls


@pytest.mark.parametrize("seed", range(6))
def test_restatement_matches_brute_force(seed):
    rng = np.random.RandomState(seed)
    n, d = rng.randint(20, 120), rng.randint(5, 60)
    X = sp.random(n, d, density=rng.uniform(0.02, 0.15), random_state=seed, format="csr")
    X.data = rng.randn(X.nnz)
    order = rng.permutation(d) if seed % 2 else np.arange(d)
    for B in (1, 2, 3, 7, d - 1, d, d + 3):
        if B < 1:
            continue
        for H in (0, 1):
            for near in (0, 1, 2):
                p = M.Plan(X, order, B, H, near, slot_cap=1 << 20)
                hot, slots, ht_cls = _brute(X, order, B, H, near)
                assert np.array_equal(p.hot, hot), (B, H)
                assert [s.tolist() for s in p.slots] == slots, (B, H)
                assert np.array_equal(p.n_slots, [len(s) for s in slots])
                assert np.array_equal(p.ht_cls, ht_cls), (B, H, near)
                assert np.array_equal(p.hot_count, [len(e) for e in p.ent])
                # entries in class order; dep is the last earlier toucher inside the window
                for t, es in enumerate(p.ent):
                    cls = [0 if lt and not fw else 1 if lt else 2 if fw else 3 for _, _, lt, fw, _ in es]
                    assert cls == sorted(cls)
                    for i, dep, lt, fw, x in es:
                        w0 = (t // B) * B
                        assert dep < t - w0 and (dep == -1 or i in [r[0] for r in p.ent[w0 + dep]])


def test_small_cases_by_hand():
    # sample 0 at columns 0 and 2, sample 1 at column 1 only, sample 2 at columns 1 and 5
    X = sp.csr_matrix((np.ones(5), [0, 2, 1, 1, 5], [0, 2, 3, 5]), shape=(3, 6))
    p = M.window_plan(X, 3, 0, 2, slot_cap=8)
    assert p.hot.tolist() == [True, False, False, True, False]    # CSC order: (0,0) (1,1) (2,1) (0,2) (2,5)
    assert p.n_slots.tolist() == [1, 0]
    assert p.ht_cls.tolist() == [1 << 16, 0, 1, 0, 0, 0]          # fwd-only at 0, late-only at 2
    assert M.window_plan(X, 3, 0, 1, slot_cap=8).ht_cls.tolist() == [0] * 6     # distance 2 > near 1
    p1 = M.window_plan(X, 3, 1, 1, slot_cap=8)
    assert p1.hot.tolist() == [True, False, True, True, True]     # horizon 1: column 5 is a window away
    assert p1.n_slots.tolist() == [2, 1]
    assert M.window_plan(X, 2, 0, 1, slot_cap=8).n_slots.tolist() == [0, 0, 0]


def test_slot_caps():
    assert [M.pcd_slot_cap(s) for s in (2, 4, 8)] == [3510, 2730, 1890]
    assert M.pbcd_slot_cap(2, 32) == 531 and M.pbcd_slot_cap(3, 32) == 290
    assert M.pbcd_slot_cap(2, 8) == 1412 and M.pbcd_slot_cap(2, 33) == 0


def _background(n=4000, d=960, r=4, seed=0):
    from sparsepoly_b200 import synth
    return synth.uniform_sparse(n, d, r, seed)


@pytest.mark.parametrize("cap,ent,H,B,n", [(M.pcd_slot_cap(4), M.PCD_ENT_PER_SLOT, 0, 96, 4000),
                                           (M.pcd_slot_cap(8), M.PCD_ENT_PER_SLOT, 1, 96, 4000),
                                           (M.pbcd_slot_cap(3, 32), M.PBCD_ENT_PER_SLOT, 1, 48, 1500)])
def test_slot_constructor_lands_on_cap(cap, ent, H, B, n):
    X = _background(n=n, r=3)
    w = 3
    for target, over in ((cap - 1, False), (cap, False), (cap + 1, True)):
        Xs = M.with_slots(X, B, H, w, target, seed=1, slot_cap=cap, ent_per_slot=ent)
        p = M.window_plan(Xs, B, H, 0, cap, ent)
        assert p.n_slots[w] == target and p.max_slots == target
        assert p.overflow == over
        assert (p.chain <= 32).all()
        assert np.delete(p.n_slots, w).max() < cap // 2
        if H == 0 and target == cap and ent == M.PCD_ENT_PER_SLOT:
            assert p.n_ent[w] == p.ent_cap                # at horizon 0 a pcd window at its slot cap is at its entry cap


@pytest.mark.parametrize("near", [1, 2])
@pytest.mark.parametrize("n_late,n_both,n_fwd,lanes", [(16, 0, 15, 31), (16, 0, 16, 32), (11, 10, 11, 32),
                                                       (17, 0, 16, 33)])
def test_chain_constructor_lands_on_lanes(n_late, n_both, n_fwd, lanes, near):
    X = _background()
    B, t = 96, 96 * 4 + 40
    Xc = M.with_chain(X, t, n_late, n_both, n_fwd, near, seed=2)
    p = M.window_plan(Xc, B, 0, near, M.pcd_slot_cap(4))
    assert p.chain[t] == lanes
    assert p.ht_cls[t] == n_late | (n_both << 8) | (n_fwd << 16)
    assert p.chain.max() == lanes
    assert p.overflow == (lanes > 32)
    assert M.built_near(Xc, B, 0, near, M.pcd_slot_cap(4)) == (near if lanes <= 32 else 0)
    # at near = dist - 1 the pairs are too far apart to be late
    if near > 1:
        assert M.window_plan(Xc, B, 0, near - 1, M.pcd_slot_cap(4)).chain[t] == 0


def test_full_chain_and_cold_window_constructors():
    X = _background()
    B, w = 96, 2
    Xf = M.with_full_chain(X, w, B, seed=3)
    p = M.window_plan(Xf, B, 0, 1, M.pcd_slot_cap(4))
    last = Xf.shape[0] - 1
    deps = [[dep for i, dep, *_ in p.ent[w * B + tl] if i == last] for tl in range(B)]
    assert deps == [[tl - 1] for tl in range(B)]
    Xn = M.without_hot(X, B, 1, w)
    p = M.window_plan(Xn, B, 1, 1, M.pcd_slot_cap(4))
    assert p.n_slots[w] == 0 and p.hot_count[w * B:(w + 1) * B].sum() == 0
    assert p.n_slots[w + 1] > 0
