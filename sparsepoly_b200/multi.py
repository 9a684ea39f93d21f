"""fit_many: fit many pcd or pbcd models on one design matrix at once (DESIGN.md 3.2 / 3.3, "Many models per
launch").

A pcd or pbcd fit is one sequential coordinate chain and, at the sizes the reference is used at (hyper-parameter
grids, one-vs-rest classes, gamma sweeps of the feature-selecting regularizers), one chain fills a single
thread-block cluster of the GPU.  fit_many runs the chains of many models side by side: every launch of an epoch
covers all models still running, one cluster (one row-DP block row, one regularizer-cache block) per model.  Each
cluster runs the code a single fit runs on that model's own records, so every model ends bit-identical to
``est.fit(X, y_i)`` run alone with the cluster sweep (SPARSEPOLY_B200_SWEEP=cluster) and the same geometry.
"""
import contextlib
import ctypes as C
import io
import numbers
import warnings

import numpy as np
import torch
import scipy.sparse as sp
from sklearn.utils import check_random_state

from . import _lib, solvers
from .dataset import DeviceDataset, SweepPlan, _device, choose_geometry
from .estimators import _BaseSparseAllSubsets, _BaseSparseFactorizationMachine

_f64 = torch.float64

# parameters that fix the kernel instantiation, the shape of P and the augmented X: equal across a call
_SHARED_FM = ("degree", "n_components", "loss", "fit_lower", "fit_linear")
_SHARED_ALL = ("n_components", "loss")


def _targets(y, n_models):
    """One target per model: y itself, or the elements of a sequence of arrays."""
    if isinstance(y, (list, tuple)) and len(y) > 0 and all(np.ndim(t) >= 1 for t in y):
        if len(y) != n_models:
            raise ValueError(f"fit_many: {len(y)} target arrays for {n_models} estimators")
        return list(y)
    return [y] * n_models


def _check_generators(ests):
    """A shuffling model draws every epoch; its draws only come out as in a sequential fit when nobody else
    draws from its generator in between.  None means numpy's global generator, which counts as shared."""
    def key(rs):
        if rs is None or rs is np.random.mtrand._rand:
            return "numpy global"
        if isinstance(rs, numbers.Integral):
            return None                                   # a fresh generator per fit
        return id(rs)
    keys = [key(e.random_state) for e in ests]
    for i, e in enumerate(ests):
        if e.shuffle and keys[i] is not None and (keys[i] == "numpy global" or keys.count(keys[i]) > 1):
            raise ValueError(f"fit_many: estimator {i} has shuffle=True and shares its random generator "
                             f"(random_state={e.random_state!r}); give it an int or its own RandomState")


SOLVERS = ("pcd", "pbcd")
PBCD_MAX_COMPONENTS = 128          # widest component block of the pbcd sweep (KCH = 4)


def _validate(ests):
    """Every check of a fit_many call that needs no device: returns (fm, solver)."""
    first = ests[0]
    if not isinstance(first, (_BaseSparseFactorizationMachine, _BaseSparseAllSubsets)):
        raise ValueError(f"fit_many: {type(first).__name__} is not a SparseFactorizationMachine or "
                         "SparseAllSubsets estimator")
    fm = isinstance(first, _BaseSparseFactorizationMachine)
    solver = first.solver
    if solver not in SOLVERS:
        raise ValueError(f"fit_many: estimator 0 has solver={solver!r}; fit_many supports solver='pcd' or "
                         "solver='pbcd'")
    for i, e in enumerate(ests):
        if e.solver != solver:
            raise ValueError(f"fit_many: estimator {i} has solver={e.solver!r}; a call whose first estimator has "
                             f"solver={solver!r} supports solver={solver!r} only")
        if type(e) is not type(first):
            raise ValueError(f"fit_many: estimator {i} is a {type(e).__name__} and estimator 0 a "
                             f"{type(first).__name__}; all estimators must be of one class")
        for name in (_SHARED_FM if fm else _SHARED_ALL):
            if getattr(e, name) != getattr(first, name):
                raise ValueError(f"fit_many: {name} must be equal across the estimators "
                                 f"(estimator {i}: {getattr(e, name)!r}, estimator 0: {getattr(first, name)!r})")
        e._get_loss(e.loss)
        e._get_regularizer(e.regularizer)
        e._check_combination(solver, e.regularizer, e.degree if fm else -1)
        if not (e.warm_start and hasattr(e, "lams_")) and e.init_lambdas not in ("ones", "random_signs"):
            e._init_lambdas(None)                         # raises the estimator's own ValueError
    if fm and not 2 <= first.degree <= 5:
        raise ValueError(f"fit_many: {solver} degree {first.degree} is not supported by the CUDA backend (2..5)")
    if solver == "pbcd" and first.n_components > PBCD_MAX_COMPONENTS:
        raise ValueError(f"fit_many: pbcd n_components={first.n_components} > {PBCD_MAX_COMPONENTS} is not "
                         "supported by the CUDA backend")
    _check_generators(ests)
    return fm, solver


def _pbcd_bytes(ests, n, d, nnz, fm):
    """(shared, per model, per shuffling model's plan) device bytes of a pbcd call.  A model holds its A cache
    (n·(m−1)·k doubles, n·k for all-subsets), P twice (as uploaded and feature-major), w, lams, {y_pred, y} per
    sample and O(d) regularizer scratch; the plan bound is that of the widest cluster (16 CTAs)."""
    first = ests[0]
    k = first.n_components
    if fm:
        n_orders = first.degree - 1 if first.fit_lower == "explicit" else 1
        a = n * (first.degree - 1) * k
    else:
        n_orders, a = 1, n * k
    plan = 4 * (2 * d * 17 + nnz + 2 * d)                  # col_part, pos_ptr, flag_idx, pos_conf, idx_feat
    shared = 2 * (12 * nnz) + 4 * (n + d + 2) + 8 * d + plan   # CSR + CSC, col_norm_sq, the unshuffled plan
    model = 8 * (max(a, 1) + 2 * n + 2 * n_orders * d * k + 2 * d + k + 17)
    return shared, model, plan


def _free_device_bytes():
    """Free device memory, counting what PyTorch's caching allocator holds but does not use."""
    dev = _device()
    free, _ = torch.cuda.mem_get_info(dev)
    return free + torch.cuda.memory_reserved(dev) - torch.cuda.memory_allocated(dev)


def _check_memory(ests, n, d, nnz, fm):
    shared, model, plan = _pbcd_bytes(ests, n, d, nnz, fm)
    need = shared + len(ests) * model + sum(plan for e in ests if e.shuffle)
    free = _free_device_bytes()
    if need > free:
        per = (need - shared) / len(ests)               # a model, with this call's share of shuffling plans
        fit = max(0, int((free - shared) // per))
        raise ValueError(f"fit_many: {len(ests)} pbcd models need {need / 2**30:.2f} GiB of device memory and "
                         f"{free / 2**30:.2f} GiB are free; {fit} models of this shape fit at a time "
                         f"({model / 2**20:.1f} MiB per model, mostly its A cache of n*(degree-1)*n_components "
                         "doubles): split the call")


class _Model:
    """Device state and stopping state of one model of a fit_many call."""

    def __init__(self, b, est, rng, y, ds, plan, stride, fm, pbcd, dev):
        self.b, self.est, self.rng, self.plan = b, est, rng, plan
        self.fm, self.pbcd = fm, pbcd
        n, d = ds.n_samples, ds.n_features
        self.rec = torch.zeros(n * stride, dtype=_f64, device=dev)
        self.rec[1::stride] = torch.from_numpy(y).to(dev)
        self.P = torch.from_numpy(np.ascontiguousarray(est.P_)).to(dev)
        self.lams = torch.from_numpy(np.ascontiguousarray(est.lams_, dtype=np.float64)).to(dev)
        if fm:
            self.w = torch.from_numpy(np.ascontiguousarray(est.w_)).to(dev)
            est._device_output(ds, self.P, self.w, self.lams, self.rec, stride)          # y_pred -> rec[0::stride]
            self.alpha, self.beta, self.gamma = est._scaled(n)
        else:
            self.w = None
            solvers.poly_predict(ds, solvers.transpose(self.P), self.lams, -1, out=self.rec, out_stride=stride)
            self.alpha = 0.0
            self.beta, self.gamma = (n * est.beta, n * est.gamma) if est.mean else (est.beta, est.gamma)
        self.regstate = torch.zeros(16, dtype=_f64, device=dev)
        self.idx_feat = np.arange(d, dtype=np.int32)
        self.idx_comp = None
        if pbcd:                    # the feature-major copy and scratch of _pbcd_setup / _setup
            k = est.n_components
            if fm:
                self.P = torch.stack([solvers.transpose(self.P[o]) for o in range(self.P.shape[0])])
                self.A = torch.empty(max(n * (est.degree - 1) * k, 1), dtype=_f64, device=dev)
            else:
                self.P = solvers.transpose(self.P)
                self.A = torch.empty(max(n * k, 1), dtype=_f64, device=dev)
            self.reg_norms = torch.zeros(max(d, 1), dtype=_f64, device=dev)
        else:
            self.idx_comp = np.arange(est.n_components, dtype=np.int32)
        self.it, self.converged, self.out = 0, False, io.StringIO()

    def shuffle(self):
        """The draws of one epoch: pcd shuffles the components then the features, pbcd the features only."""
        if self.idx_comp is not None:
            self.rng.shuffle(self.idx_comp)
        self.rng.shuffle(self.idx_feat)
        self.plan.set_order(self.idx_feat)

    def sync(self):
        if not self.pbcd:
            self.est.P_[...] = self.P.cpu().numpy()
        elif self.fm:
            for o in range(self.P.shape[0]):
                self.est.P_[o] = solvers.transpose(self.P[o]).cpu().numpy()
        else:
            self.est.P_[...] = solvers.transpose(self.P).cpu().numpy()
        if self.w is not None:
            self.est.w_[...] = self.w.cpu().numpy()

    def descriptor(self, P, ab, viol):
        s = self.plan.struct
        idx_comp = None if self.idx_comp is None else self.idx_comp.ctypes.data_as(C.POINTER(C.c_int32))
        return _lib.SpPcdModel(pos_ptr=s.pos_ptr, flag_idx=s.flag_idx, idx_feat=s.idx_feat, pos_conf=s.pos_conf,
                               P=P.data_ptr(), lams=self.lams.data_ptr(), ab=float(ab), gamma=float(self.gamma),
                               eta=float(self.est.eta0), reg=_lib.REG_IDS[self.est.regularizer],
                               rec=self.rec.data_ptr(), regstate=self.regstate.data_ptr(),
                               viol=viol.data_ptr() + 8 * self.b, idx_comp_host=idx_comp)

    def pbcd_descriptor(self, P, viol):
        s = self.plan.struct
        return _lib.SpPbcdModel(pos_ptr=s.pos_ptr, flag_idx=s.flag_idx, idx_feat=s.idx_feat, P=P.data_ptr(),
                                lams=self.lams.data_ptr(), beta=float(self.beta), gamma=float(self.gamma),
                                eta=float(self.est.eta0), reg=_lib.REG_IDS[self.est.regularizer],
                                yrec=self.rec.data_ptr(), A=self.A.data_ptr(), reg_norms=self.reg_norms.data_ptr(),
                                regstate=self.regstate.data_ptr(), viol=viol.data_ptr() + 8 * self.b)


def _descriptors(models, P_of, ab_of, viol):
    arr = (_lib.SpPcdModel * len(models))()
    for i, m in enumerate(models):
        arr[i] = m.descriptor(P_of(m), ab_of(m), viol)
    return arr


def _pbcd_descriptors(models, P_of, viol):
    arr = (_lib.SpPbcdModel * len(models))()
    for i, m in enumerate(models):
        arr[i] = m.pbcd_descriptor(P_of(m), viol)
    return arr


def fit_many(estimators, X, y):
    """Fit many pcd or pbcd estimators on one design matrix X at once; returns them (fitted in place) as a list.

    estimators: SparseFactorizationMachine{Regressor,Classifier} or SparseAllSubsets{Regressor,Classifier}
    instances, all of one class and one solver ("pcd" or "pbcd", as the first estimator has it) and with equal
    degree, n_components, loss, fit_lower and fit_linear.  regularizer, alpha, beta, gamma, eta0, mean, tol,
    max_iter, shuffle, warm_start, init_lambdas, random_state, verbose, callback and n_calls may differ.  A model
    with shuffle=True needs an int or a RandomState of its own as random_state.  pbcd takes n_components <= 128.
    y: one target array for every model, or a sequence of one target array per estimator (one-vs-rest).

    Each estimator's P_, w_, lams_, n_iter_, label_binarizer_, convergence warning, verbose lines and callback
    calls are those of est.fit(X, y_i) alone with SPARSEPOLY_B200_SWEEP=cluster.  A model stops as fit would
    (violation below tol, callback returning non-None, max_iter); later launches cover the others only.  Its
    verbose lines are printed when the call returns, model by model in list order.

    Device memory: a pbcd model holds its A cache of n_samples·(degree−1)·n_components doubles
    (n_samples·n_components for all-subsets), P twice, w, lams, two doubles per sample and O(n_features) scratch,
    all for the whole call; a shuffling model also its own coordinate plan.  When the call would not fit in the
    free device memory it raises ValueError, naming how many models of that shape fit, before anything is drawn.
    """
    ests = list(estimators)
    if not ests:
        return []
    fm, solver = _validate(ests)
    pbcd = solver == "pbcd"
    first = ests[0]
    checked = [e._check_X_y(X, yi) for e, yi in zip(ests, _targets(y, len(ests)))]
    Xc = checked[0][0]
    if fm:
        Xc = first._augment(Xc)
    n, d = Xc.shape
    degree = first.degree if fm else -1
    k, loss = first.n_components, first.loss
    if pbcd:
        _check_memory(ests, n, d, Xc.nnz if sp.issparse(Xc) else n * d, fm)

    dev = _device()
    _lib.check(_lib.load().sp_set_device(dev.index if dev.index is not None else 0))
    rngs = [check_random_state(e.random_state) for e in ests]
    for e, rng in zip(ests, rngs):                # the draws of sequential fits, in list order
        e._init_coefs(d, rng)

    stride = 2 if pbcd else solvers.rec_stride(degree)
    ds = DeviceDataset(Xc, need_csr=True, need_csc=True, device=dev)

    def new_plan():
        plan = SweepPlan(ds, solver, rec_stride=None if pbcd else stride, sweep="cluster")
        plan.set_order(np.arange(d, dtype=np.int32))
        return plan

    plan0 = new_plan()                            # the unshuffled models' order
    n_cta, threads = plan0.n_cta, plan0.threads
    # pbcd's linear sub-epoch runs the pcd sweep at the pcd geometry (same n_cta, its own threads) on the
    # model's plan: pos_ptr / flag_idx / pos_conf depend on the order and n_cta only
    threads_lin = choose_geometry(ds, "pcd")[1] if pbcd else threads
    col_norm_sq = ds.col_norm_sq()
    viol = torch.zeros(len(ests), dtype=_f64, device=dev)
    models = []
    for b, (e, rng, (_, yb)) in enumerate(zip(ests, rngs, checked)):
        plan = new_plan() if e.shuffle else plan0
        models.append(_Model(b, e, rng, np.ascontiguousarray(yb, dtype=np.float64), ds, plan, stride, fm, pbcd,
                             dev))

    def epoch_orders(active):
        """The per-epoch order of _pcd_setup / _pbcd_setup / _setup: linear CD -> explicit lower orders
        ascending -> top order."""
        if fm and first.fit_linear:
            solvers.cd_linear_epoch_multi(ds, n_cta, threads_lin, col_norm_sq,
                                          _descriptors(active, lambda m: m.w, lambda m: m.alpha, viol), loss, stride)
        top = (lambda m: m.P[0]) if fm else (lambda m: m.P)
        orders = [(deg, lambda m, deg=deg: m.P[degree - deg])
                  for deg in (range(2, degree) if fm and first.fit_lower == "explicit" else ())]
        for deg, P_of in orders + [(degree, top)]:
            if pbcd:
                solvers.pbcd_epoch_multi(ds, n_cta, threads, _pbcd_descriptors(active, P_of, viol), k, deg, loss)
            else:
                solvers.pcd_epoch_multi(ds, n_cta, threads, _descriptors(active, P_of, lambda m: m.beta, viol),
                                        k, deg, loss, stride)

    active = [m for m in models if m.est.max_iter > 0]
    it = 0
    while active:
        viol.zero_()
        for m in active:
            if m.est.shuffle:
                m.shuffle()
        epoch_orders(active)
        v = viol.cpu().numpy()
        running = []
        for m in active:
            e = m.est
            m.it = it
            with contextlib.redirect_stdout(m.out):
                stop = e._after_epoch(it, float(v[m.b]), "Iteration {} violation sum {}", m.sync)
                if not stop and float(v[m.b]) < e.tol:
                    if e.verbose:
                        print(f"Converged at iteration {it+1}")
                    m.converged = stop = True
            if not stop and it + 1 < e.max_iter:
                running.append(m)
        active = running
        it += 1

    for m in models:
        m.sync()
        m.est.n_iter_ = m.it
        print(m.out.getvalue(), end="")
        if not m.converged:
            warnings.warn("Objective did not converge. Increase max_iter.")
    return ests
