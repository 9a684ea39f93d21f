"""Host restatement of the window plan of the pipelined sweeps (csrc/wplan.cu, DESIGN.md §2) and input
constructors that put one window of that plan exactly at a limit of the engine CTA.

The plan, for CSR X, a coordinate order (position t visits column order[t]), window B, horizon H and `near`:
  * a nonzero (sample i, column j) is HOT when sample i has another nonzero in a column whose window is within H
    windows of j's window;
  * the slots of window w are the distinct samples of the window's hot nonzeros;
  * walking the window's positions in order, a hot nonzero's `dep` is the window-local position that last touched
    its sample (-1: none); it is LATE when dep >= 0 and (position - dep) <= near, and then the nonzero of `dep`
    that touched the sample is marked FWD;
  * ht_cls[t] = #late-only | #late+fwd << 8 | #fwd-only << 16: these go to the chain warp, one per lane;
  * the plan overflows when a window needs more than slot_cap slots or more than ent_per_slot * slot_cap hot
    nonzeros, or a position more than 32 chain-warp lanes.
WindowPlan.build retries an overflowing window with near = 0 before it gives up on the window size.

Without shuffling the estimators visit position t = column t, so the constructors place nonzeros by column index.
"""
import numpy as np
import scipy.sparse as sp

CHAIN_LANES = 32                 # one chain-warp lane per late / fwd nonzero of a position
PCD_WINDOW_MAX = 256             # SP_WINDOW_MAX
PBCD_WINDOW_MAX = 64             # BWIN of pbcd_window.cu
SPEC_WINDOW_MAX = 128            # 128-bit known-mover masks: a pcd window speculates only when nb <= 128
PCD_ENT_PER_SLOT = 2
PBCD_ENT_PER_SLOT = 3            # SP_PBCD_ENT_PER_SLOT


def pcd_slot_cap(rec_stride):
    """sp_wplan_slot_cap: 196 608 bytes of slots, each a record, two hot nonzeros (12 B each) and a 128-bit
    mover mask; even."""
    return min(8192, (196608 // (max(rec_stride, 2) * 8 + 40)) & ~1)


def pbcd_slot_cap(degree, k):
    """sp_pbcd_wplan_slot_cap: 160 KiB of slots, each A[i, :, :] + {y_pred, y} padded to an even count of
    doubles, and three hot nonzeros."""
    if not 1 <= k <= 32:
        return 0
    na = 1 if degree == -1 else degree - 1
    slotsz = (na * k + 3) & ~1
    return min(8192, 163840 // (slotsz * 8 + 12 * PBCD_ENT_PER_SLOT))


class Plan:
    """The restated plan.  Arrays follow the library's: hot[e] per CSC nonzero (canonical CSC of X), hot_count /
    ht_cls / chain per position, n_slots / n_ent per window, slots[w] = sorted sample ids, ent[t] = the position's
    hot nonzeros as (sample, dep, late, fwd, value) in the class order of h_sd."""

    def __init__(self, X, order, B, H, near, slot_cap, ent_per_slot=PCD_ENT_PER_SLOT):
        X = sp.csr_matrix(X)
        d = X.shape[1]
        order = np.asarray(order, dtype=np.int64)
        self.B, self.H, self.near, self.slot_cap = B, H, near, slot_cap
        self.ent_cap = ent_per_slot * slot_cap
        self.n_windows = (d + B - 1) // B
        pos = np.empty(d, dtype=np.int64)
        pos[order] = np.arange(d)
        Xc = sp.csc_matrix(X)
        Xc.sort_indices()
        rows = Xc.indices.astype(np.int64)
        cols = np.repeat(np.arange(d), np.diff(Xc.indptr))
        win = pos[cols] // B
        # per nonzero: how many nonzeros its sample has in each window near its own
        stride = self.n_windows + 2
        key = rows * stride + win + 1
        srt = np.sort(key)

        def count(k):
            return np.searchsorted(srt, k, "right") - np.searchsorted(srt, k, "left")

        others = count(key) - 1
        if H >= 1:
            others = others + count(key - 1) + count(key + 1)
        self.hot = others > 0
        self.hot_count = np.zeros(d, dtype=np.int64)
        np.add.at(self.hot_count, pos[cols[self.hot]], 1)
        self.n_slots = np.zeros(self.n_windows, dtype=np.int64)
        self.n_ent = np.zeros(self.n_windows, dtype=np.int64)
        self.slots = []
        self.ht_cls = np.zeros(d, dtype=np.int64)
        self.chain = np.zeros(d, dtype=np.int64)
        self.ent = [[] for _ in range(d)]
        for w in range(self.n_windows):
            t0, nb = w * B, min(B, d - w * B)
            last = {}                      # sample -> (window-local position, entry) of its last hot nonzero
            window_ent = []
            for tl in range(nb):
                j = order[t0 + tl]
                lo, hi = Xc.indptr[j], Xc.indptr[j + 1]
                for e in range(lo, hi):
                    if not self.hot[e]:
                        continue
                    i = int(rows[e])
                    dep, prev = last.get(i, (-1, None))
                    rec = [i, dep, dep >= 0 and tl - dep <= near, False, float(Xc.data[e])]
                    if rec[2]:
                        prev[3] = True
                    last[i] = (tl, rec)
                    self.ent[t0 + tl].append(rec)
                    window_ent.append(rec)
            self.slots.append(np.array(sorted(last), dtype=np.int64))
            self.n_slots[w] = len(last)
            self.n_ent[w] = len(window_ent)
            for tl in range(nb):
                t = t0 + tl
                es = self.ent[t]
                cls = [0 if r[2] and not r[3] else 1 if r[2] else 2 if r[3] else 3 for r in es]
                self.ent[t] = [tuple(r) for c in range(4) for r, k in zip(es, cls) if k == c]
                cnt = [cls.count(c) for c in range(3)]
                self.ht_cls[t] = cnt[0] | (cnt[1] << 8) | (cnt[2] << 16)
                self.chain[t] = sum(cnt)

    @property
    def max_slots(self):
        return int(self.n_slots.max()) if self.n_slots.size else 0

    @property
    def overflow(self):
        return bool((self.n_slots > self.slot_cap).any() or (self.n_ent > self.ent_cap).any()
                    or (self.chain > CHAIN_LANES).any())


def window_plan(X, B, H, near, slot_cap, ent_per_slot=PCD_ENT_PER_SLOT, order=None):
    """Plan of the identity order (the estimators' order without shuffling) unless `order` is given."""
    return Plan(X, np.arange(X.shape[1]) if order is None else order, B, H, near, slot_cap, ent_per_slot)


def built_near(X, B, H, near, slot_cap, ent_per_slot=PCD_ENT_PER_SLOT, order=None):
    """The `near` WindowPlan.build settles on for a forced window B (near, then 0), or None when neither fits."""
    for nr in ((near, 0) if near > 0 else (0,)):
        if not window_plan(X, B, H, nr, slot_cap, ent_per_slot, order).overflow:
            return nr
    return None


# ------------------------------------------------------------------------------------------ input constructors
def _rows(entries, d):
    """CSR of rows given as lists of (column, value)."""
    indptr = np.cumsum([0] + [len(r) for r in entries])
    cols = np.array([c for r in entries for c, _ in r], dtype=np.int64)
    vals = np.array([v for r in entries for _, v in r], dtype=np.float64)
    X = sp.csr_matrix((vals, cols, indptr), shape=(len(entries), d))
    X.sort_indices()
    return X


def _drop_columns(X, cols):
    X = sp.csr_matrix(X, copy=True)
    keep = ~np.isin(X.indices, np.asarray(cols))
    X.data = np.where(keep, X.data, 0.0)
    X.eliminate_zeros()
    return X


def with_slots(X, B, H, w, target, seed, slot_cap, ent_per_slot=PCD_ENT_PER_SLOT):
    """X plus "pair" samples, each with two nonzeros in columns of window w at least 3 positions apart (so no
    chain-warp lane changes), until window w has exactly `target` slots.  A sample of X keeps at most two
    nonzeros in window w, so the window holds at most 2 hot nonzeros per slot: at horizon 0 exactly two, which
    puts a pcd window at its entry cap (2 * slot_cap) too when target == slot_cap."""
    d = X.shape[1]
    t0, nb = w * B, min(B, d - w * B)
    assert nb >= 4, "a pair needs two columns at least 3 positions apart"
    X = sp.csr_matrix(X, copy=True)
    X.sort_indices()
    inw = (X.indices >= t0) & (X.indices < t0 + nb)
    c = np.concatenate([[0], np.cumsum(inw)])
    rank = c[1:] - c[np.repeat(X.indptr[:-1], np.diff(X.indptr))]        # 1-based rank inside the row's window-w run
    X.data = np.where(inw & (rank > 2), 0.0, X.data)
    X.eliminate_zeros()
    base = window_plan(X, B, H, 0, slot_cap, ent_per_slot).n_slots[w]
    need = int(target - base)
    assert need >= 0, (target, base)
    rng = np.random.RandomState(seed)
    pairs = []
    while len(pairs) < need:
        a, b = rng.randint(0, nb, size=2)
        if abs(int(a) - int(b)) > 2:
            pairs.append([(t0 + int(a), rng.randn()), (t0 + int(b), rng.randn())])
    out = sp.vstack([X, _rows(pairs, d)]).tocsr() if pairs else sp.csr_matrix(X)
    plan = window_plan(out, B, H, 0, slot_cap, ent_per_slot)
    assert plan.n_slots[w] == target, (plan.n_slots[w], target)
    return out


def with_chain(X, t, n_late, n_both, n_fwd, dist, seed):
    """X with the columns t - 2*dist .. t + 2*dist cleared and then touched only by samples that make position t
    hand exactly n_late + n_both + n_fwd nonzeros to the chain warp at near = dist: n_late samples with nonzeros
    at t - dist and t (late only at t), n_fwd at t and t + dist (fwd only), n_both at t - dist, t, t + dist (late
    and fwd).  Positions t - dist .. t + dist must lie in one window."""
    d = X.shape[1]
    assert t - 2 * dist >= 0 and t + 2 * dist < d
    X = _drop_columns(X, np.arange(t - 2 * dist, t + 2 * dist + 1))
    rng = np.random.RandomState(seed)
    rows = ([[(t - dist, rng.randn()), (t, rng.randn())] for _ in range(n_late)]
            + [[(t - dist, rng.randn()), (t, rng.randn()), (t + dist, rng.randn())] for _ in range(n_both)]
            + [[(t, rng.randn()), (t + dist, rng.randn())] for _ in range(n_fwd)])
    return sp.vstack([X, _rows(rows, d)]).tocsr()


def with_full_chain(X, w, B, seed):
    """X plus one sample with a nonzero in every column of window w: every position of the window depends on
    the one before it (the longest dependency chain a window can have)."""
    d = X.shape[1]
    t0, nb = w * B, min(B, d - w * B)
    rng = np.random.RandomState(seed)
    return sp.vstack([X, _rows([[(t0 + tl, rng.randn()) for tl in range(nb)]], d)]).tocsr()


def without_hot(X, B, H, w):
    """X without the nonzeros of window w that are hot: no sample of window w has another nonzero within H
    windows, so the window has no slot and its whole reduction runs in the bulk CTAs."""
    plan = window_plan(X, B, H, 0, 1 << 30)
    Xc = sp.csc_matrix(X)
    Xc.sort_indices()
    d = X.shape[1]
    cols = np.repeat(np.arange(d), np.diff(Xc.indptr))
    drop = plan.hot & (cols // B == w)
    Xc = Xc.copy()
    Xc.data = np.where(drop, 0.0, Xc.data)
    Xc.eliminate_zeros()
    out = sp.csr_matrix(Xc)
    out.sort_indices()
    assert window_plan(out, B, H, 0, 1 << 30).n_slots[w] == 0
    return out
