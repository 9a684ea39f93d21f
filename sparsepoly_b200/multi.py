"""fit_many: fit many pcd models on one design matrix at once (DESIGN.md 3.2, "Many models per launch").

A pcd fit is one sequential coordinate chain and, at the sizes the reference is used at (hyper-parameter
grids, one-vs-rest classes), one chain fills a single thread-block cluster of the GPU.  fit_many runs the
chains of many models side by side: every launch of an epoch covers all models still running, one cluster
(one row-DP block row, one regularizer-cache block) per model.  Each cluster runs the code a single fit runs
on that model's own records, so every model ends bit-identical to ``est.fit(X, y_i)`` run alone with the
cluster sweep (SPARSEPOLY_B200_SWEEP=cluster) and the same geometry.
"""
import contextlib
import ctypes as C
import io
import numbers
import warnings

import numpy as np
import torch
from sklearn.utils import check_random_state

from . import _lib, solvers
from .dataset import DeviceDataset, SweepPlan, _device
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


def _validate(ests):
    first = ests[0]
    if not isinstance(first, (_BaseSparseFactorizationMachine, _BaseSparseAllSubsets)):
        raise ValueError(f"fit_many: {type(first).__name__} is not a SparseFactorizationMachine or "
                         "SparseAllSubsets estimator")
    fm = isinstance(first, _BaseSparseFactorizationMachine)
    for i, e in enumerate(ests):
        if e.solver != "pcd":
            raise ValueError(f"fit_many: estimator {i} has solver={e.solver!r}; fit_many supports solver='pcd' only")
        if type(e) is not type(first):
            raise ValueError(f"fit_many: estimator {i} is a {type(e).__name__} and estimator 0 a "
                             f"{type(first).__name__}; all estimators must be of one class")
        for name in (_SHARED_FM if fm else _SHARED_ALL):
            if getattr(e, name) != getattr(first, name):
                raise ValueError(f"fit_many: {name} must be equal across the estimators "
                                 f"(estimator {i}: {getattr(e, name)!r}, estimator 0: {getattr(first, name)!r})")
        e._get_loss(e.loss)
        e._get_regularizer(e.regularizer)
        e._check_combination("pcd", e.regularizer, e.degree if fm else -1)
        if not (e.warm_start and hasattr(e, "lams_")) and e.init_lambdas not in ("ones", "random_signs"):
            e._init_lambdas(None)                         # raises the estimator's own ValueError
    if fm and not 2 <= first.degree <= 5:
        raise ValueError(f"fit_many: pcd degree {first.degree} is not supported by the CUDA backend (2..5)")
    _check_generators(ests)
    return fm


class _Model:
    """Device state and stopping state of one model of a fit_many call."""

    def __init__(self, b, est, rng, y, ds, plan, stride, fm, dev):
        self.b, self.est, self.rng, self.plan = b, est, rng, plan
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
        self.idx_comp = np.arange(est.n_components, dtype=np.int32)
        self.it, self.converged, self.out = 0, False, io.StringIO()

    def sync(self):
        self.est.P_[...] = self.P.cpu().numpy()
        if self.w is not None:
            self.est.w_[...] = self.w.cpu().numpy()

    def descriptor(self, P, ab, viol):
        s = self.plan.struct
        return _lib.SpPcdModel(pos_ptr=s.pos_ptr, flag_idx=s.flag_idx, idx_feat=s.idx_feat, pos_conf=s.pos_conf,
                               P=P.data_ptr(), lams=self.lams.data_ptr(), ab=float(ab), gamma=float(self.gamma),
                               eta=float(self.est.eta0), reg=_lib.REG_IDS[self.est.regularizer],
                               rec=self.rec.data_ptr(), regstate=self.regstate.data_ptr(),
                               viol=viol.data_ptr() + 8 * self.b,
                               idx_comp_host=self.idx_comp.ctypes.data_as(C.POINTER(C.c_int32)))


def _descriptors(models, P_of, ab_of, viol):
    arr = (_lib.SpPcdModel * len(models))()
    for i, m in enumerate(models):
        arr[i] = m.descriptor(P_of(m), ab_of(m), viol)
    return arr


def fit_many(estimators, X, y):
    """Fit many pcd estimators on one design matrix X at once; returns them (fitted in place) as a list.

    estimators: SparseFactorizationMachine{Regressor,Classifier} or SparseAllSubsets{Regressor,Classifier}
    instances with solver="pcd", all of one class and with equal degree, n_components, loss, fit_lower and
    fit_linear.  regularizer, alpha, beta, gamma, eta0, mean, tol, max_iter, shuffle, warm_start,
    init_lambdas, random_state, verbose, callback and n_calls may differ.  A model with shuffle=True needs an
    int or a RandomState of its own as random_state.
    y: one target array for every model, or a sequence of one target array per estimator (one-vs-rest).

    Each estimator's P_, w_, lams_, n_iter_, label_binarizer_, convergence warning, verbose lines and callback
    calls are those of est.fit(X, y_i) alone with SPARSEPOLY_B200_SWEEP=cluster.  A model stops as fit would
    (violation below tol, callback returning non-None, max_iter); later launches cover the others only.  Its
    verbose lines are printed when the call returns, model by model in list order.
    """
    ests = list(estimators)
    if not ests:
        return []
    fm = _validate(ests)
    first = ests[0]
    checked = [e._check_X_y(X, yi) for e, yi in zip(ests, _targets(y, len(ests)))]
    Xc = checked[0][0]
    if fm:
        Xc = first._augment(Xc)
    n, d = Xc.shape
    degree = first.degree if fm else -1
    k, loss = first.n_components, first.loss

    dev = _device()
    _lib.check(_lib.load().sp_set_device(dev.index if dev.index is not None else 0))
    rngs = [check_random_state(e.random_state) for e in ests]
    for e, rng in zip(ests, rngs):                # the draws of sequential fits, in list order
        e._init_coefs(d, rng)

    stride = solvers.rec_stride(degree)
    ds = DeviceDataset(Xc, need_csr=True, need_csc=True, device=dev)
    plan0 = SweepPlan(ds, "pcd", rec_stride=stride, sweep="cluster")      # the unshuffled models' order
    plan0.set_order(np.arange(d, dtype=np.int32))
    n_cta, threads = plan0.n_cta, plan0.threads
    col_norm_sq = ds.col_norm_sq()
    viol = torch.zeros(len(ests), dtype=_f64, device=dev)
    models = []
    for b, (e, rng, (_, yb)) in enumerate(zip(ests, rngs, checked)):
        plan = SweepPlan(ds, "pcd", rec_stride=stride, sweep="cluster") if e.shuffle else plan0
        if e.shuffle:
            plan.set_order(np.arange(d, dtype=np.int32))
        models.append(_Model(b, e, rng, np.ascontiguousarray(yb, dtype=np.float64), ds, plan, stride, fm, dev))

    active = [m for m in models if m.est.max_iter > 0]
    it = 0
    while active:
        viol.zero_()
        for m in active:
            if m.est.shuffle:
                m.rng.shuffle(m.idx_comp)
                m.rng.shuffle(m.idx_feat)
                m.plan.set_order(m.idx_feat)
        # the per-epoch order of _pcd_setup / _setup: linear CD -> explicit lower orders ascending -> top order
        if fm and first.fit_linear:
            solvers.cd_linear_epoch_multi(ds, n_cta, threads, col_norm_sq,
                                          _descriptors(active, lambda m: m.w, lambda m: m.alpha, viol), loss, stride)
        if fm and first.fit_lower == "explicit":
            for deg in range(2, degree):
                solvers.pcd_epoch_multi(ds, n_cta, threads,
                                        _descriptors(active, lambda m: m.P[degree - deg], lambda m: m.beta, viol),
                                        k, deg, loss, stride)
        solvers.pcd_epoch_multi(ds, n_cta, threads,
                                _descriptors(active, (lambda m: m.P[0]) if fm else (lambda m: m.P),
                                             lambda m: m.beta, viol),
                                k, degree, loss, stride)
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
