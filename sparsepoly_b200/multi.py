"""fit_many: fit many pcd or pbcd models on one design matrix at once (DESIGN.md 3.2 / 3.3, "Many models per
launch"); decision_function_many / predict_many / score_many / objective_many: evaluate many fitted models on one
design matrix at once (DESIGN.md 3.1 / 3.5).

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
from sklearn.base import ClassifierMixin
from sklearn.exceptions import NotFittedError
from sklearn.metrics import accuracy_score, r2_score
from sklearn.utils import check_random_state

from . import _lib, objective as _objective, solvers
from .dataset import DeviceDataset, SweepPlan, _device, check_X, choose_geometry, host_y, is_device_input
from .estimators import _BaseSparseAllSubsets, _BaseSparseFactorizationMachine

_f64 = torch.float64

# parameters that fix the kernel instantiation, the shape of P and the augmented X: equal across a call
_SHARED_FM = ("degree", "n_components", "loss", "fit_lower", "fit_linear")
_SHARED_ALL = ("n_components", "loss")


def _targets(y, n_models, what="fit_many"):
    """One target per model: y itself, or the elements of a sequence of arrays."""
    if isinstance(y, (list, tuple)) and len(y) > 0 and all(np.ndim(host_y(t)) >= 1 for t in y):
        if len(y) != n_models:
            raise ValueError(f"{what}: {len(y)} target arrays for {n_models} estimators")
        return [host_y(t) for t in y]
    return [host_y(y)] * n_models


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
    ys = _targets(y, len(ests))
    checked = [first._check_X_y(X, ys[0])]
    # a CUDA X is checked and converted once; the other models take that device matrix
    X_rest = checked[0][0] if is_device_input(X) else X
    checked += [e._check_X_y(X_rest, yi) for e, yi in zip(ests[1:], ys[1:])]
    Xc = checked[0][0]
    if fm:
        Xc = first._augment(Xc)
    n, d = Xc.shape
    degree = first.degree if fm else -1
    k, loss = first.n_components, first.loss
    if pbcd:
        _check_memory(ests, n, d, Xc.nnz if hasattr(Xc, "nnz") else n * d, fm)

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


# ------------------------------------------------------------------------------ scoring many fitted models
# parameters that fix the augmented X, the output orders and the kernel instantiation: equal across a scoring call
_SCORE_SHARED_FM = ("degree", "n_components", "fit_lower", "fit_linear")
_SCORE_SHARED_ALL = ("n_components",)
SCORE_MAX_MODELS = min(_lib.PREDICT_MAX_MODELS, _lib.OBJECTIVE_MAX_ENTRIES)   # models per chunk: the kernel tables


def _validate_fitted(ests, what):
    """The checks of a scoring call that need no device: returns fm (factorization machine, not all-subsets)."""
    first = ests[0]
    if not isinstance(first, (_BaseSparseFactorizationMachine, _BaseSparseAllSubsets)):
        raise ValueError(f"{what}: {type(first).__name__} is not a SparseFactorizationMachine or SparseAllSubsets "
                         "estimator")
    fm = isinstance(first, _BaseSparseFactorizationMachine)
    for i, e in enumerate(ests):
        if type(e) is not type(first):
            raise ValueError(f"{what}: estimator {i} is a {type(e).__name__} and estimator 0 a "
                             f"{type(first).__name__}; all estimators must be of one class")
        if not hasattr(e, "P_"):
            raise NotFittedError(f"{what}: estimator {i} is not fitted.")
        for name in (_SCORE_SHARED_FM if fm else _SCORE_SHARED_ALL):
            if getattr(e, name) != getattr(first, name):
                raise ValueError(f"{what}: {name} must be equal across the estimators "
                                 f"(estimator {i}: {getattr(e, name)!r}, estimator 0: {getattr(first, name)!r})")
    return fm


def _n_dummies(est):
    """Dummy columns _augment adds (sparse_factorization_machines.py:86-92)."""
    if est.fit_lower != "augment":
        return 0
    return max(0, est.degree - (2 if est.fit_linear else 1))


def _check_X(ests, X, fm, what):
    """X as the single-model _predict checks and augments it (0 rows allowed), after the checks that the models fit
    it: every P_ of the call's shape, as wide as X after augmentation, and w_ / lams_ to match."""
    first = ests[0]
    X = check_X(X, accept_sparse=["csr", "csc"], dtype=np.double, ensure_min_samples=0)
    if fm and X.shape[0] > 0:
        X = first._augment(X)
    d = X.shape[1] + (_n_dummies(first) if fm and X.shape[0] == 0 else 0)
    k = first.n_components
    shape = ((first.degree - 1 if first.fit_lower == "explicit" else 1), k, d) if fm else (k, d)
    for i, e in enumerate(ests):
        P_shape = np.shape(e.P_)
        if P_shape[-1:] != (d,):
            raise ValueError(f"{what}: X has {d} features" + (" after augmentation" if _n_dummies(first) else "") +
                             f"; estimator {i} was fitted with {P_shape[-1] if P_shape else 0}")
        if P_shape != shape or np.shape(e.lams_) != (k,) or (fm and np.shape(e.w_) != (d,)):
            raise ValueError(f"{what}: estimator {i} has P_ {P_shape}, lams_ {np.shape(e.lams_)}"
                             + (f", w_ {np.shape(e.w_)}" if fm else "") + f"; a model of this call has P_ {shape}")
    return X, shape


def _score_bytes(n, nnz, shape, objective):
    """(shared, per model) device bytes of a scoring call: X's CSR, and per model P twice (as uploaded and
    feature-major), w, lams and its scores; objective_many adds the targets and the reduction work."""
    n_orders, k, d = shape if len(shape) == 3 else (1,) + shape
    shared = 12 * nnz + 4 * (n + 1) + 8 * d
    model = 8 * (2 * n_orders * k * d + d + k + max(n, 1))
    if objective:
        model += 8 * (max(n, 1) + solvers.reg_eval_work_doubles(d, k) + solvers.sum_work_doubles() + 8)
    return shared, model


def _chunk_size(ests, n, nnz, shape, objective, what):
    shared, model = _score_bytes(n, nnz, shape, objective)
    free = _free_device_bytes()
    fit = int((free - shared) // model) if free > shared else 0
    if fit < 1:
        raise ValueError(f"{what}: one model of this shape needs {model / 2**20:.1f} MiB of device memory next to "
                         f"X's {shared / 2**20:.1f} MiB and {free / 2**20:.1f} MiB are free")
    return max(1, min(SCORE_MAX_MODELS, fit))


class _Chunk:
    """Device state of one chunk of a scoring call: the models' P (feature-major), w, lams and scores."""

    def __init__(self, ests, fm, ds, n, shape, dev):
        first = ests[0]
        B = len(ests)
        n_orders, k, d = shape if fm else (1,) + shape
        P = torch.from_numpy(np.stack([np.asarray(e.P_, dtype=np.float64) for e in ests]).reshape(B * n_orders, k, d))
        self.P_dk = solvers.transpose_batch(P.to(dev)).view(B, n_orders, d, k)   # one H2D, one transpose launch
        self.lams = torch.from_numpy(np.stack([np.asarray(e.lams_, dtype=np.float64) for e in ests])).to(dev)
        self.w = torch.from_numpy(np.stack([np.asarray(e.w_, dtype=np.float64) for e in ests])).to(dev) if fm else None
        self.out = torch.zeros((B, max(n, 1)), dtype=_f64, device=dev)
        if n == 0:
            return
        orders = first._output_orders() if fm else [(0, -1)]
        for j, (o, deg) in enumerate(orders):          # the launches of _device_output, each over the whole chunk
            tab = (_lib.SpPredictModel * B)()
            for b in range(B):
                w = self.w[b].data_ptr() if (fm and j == 0 and first.fit_linear) else None
                tab[b] = _lib.SpPredictModel(P_dk=self.P_dk[b, o].data_ptr(), lams=self.lams[b].data_ptr(), w=w,
                                             out=self.out[b].data_ptr())
            solvers.predict_multi(ds, tab, k, deg, accumulate=j > 0)


def _prepare(ests, X, what):
    """Every check of a scoring call that needs no device: returns (fm, X checked and augmented, P_'s shape)."""
    fm = _validate_fitted(ests, what)
    Xc, shape = _check_X(ests, X, fm, what)
    return fm, Xc, shape


def _run_chunks(ests, Xc, fm, shape, what, objective=False):
    """Upload X once and yield (b0, b1, chunk) over chunks of the models that fit the device."""
    n = Xc.shape[0]
    size = _chunk_size(ests, n, Xc.nnz if hasattr(Xc, "nnz") else Xc.size, shape, objective, what)
    dev = _device()
    _lib.check(_lib.load().sp_set_device(dev.index if dev.index is not None else 0))
    ds = DeviceDataset(Xc, need_csr=True, need_csc=False, device=dev) if n > 0 else None
    for b0 in range(0, len(ests), size):
        b1 = min(len(ests), b0 + size)
        yield b0, b1, _Chunk(ests[b0:b1], fm, ds, n, shape, dev)


def decision_function_many(estimators, X):
    """Outputs of many fitted estimators on one design matrix: ndarray [n_models, n_samples] whose row b is
    estimators[b].decision_function(X) (classifiers) or estimators[b].predict(X) (regressors), bit for bit.

    estimators: fitted SparseFactorizationMachine{Regressor,Classifier} or SparseAllSubsets{Regressor,Classifier}
    instances of one class; factorization machines with equal degree, n_components, fit_lower and fit_linear,
    all-subsets models with equal n_components.  Solver, regularizer, loss, alpha / beta / gamma and mean may differ,
    and so may how P_ was obtained (any solver, partial_fit, fit_many, warm start, set by hand).

    X is checked, augmented and uploaded once; the models' P_ / w_ / lams_ go up stacked, in one copy each, and
    every output order is one launch over all models of a chunk.  Chunks hold up to SCORE_MAX_MODELS models and as
    many as the free device memory holds; results do not depend on the chunking."""
    return _decision(list(estimators), X, "decision_function_many")


def _decision(ests, X, what):
    if not ests:
        X = check_X(X, accept_sparse=["csr", "csc"], dtype=np.double, ensure_min_samples=0)
        return np.zeros((0, X.shape[0]))
    return _device_decision(ests, *_prepare(ests, X, what), what)


def _device_decision(ests, fm, Xc, shape, what):
    n = Xc.shape[0]
    out = np.empty((len(ests), n))
    for b0, b1, ch in _run_chunks(ests, Xc, fm, shape, what):
        out[b0:b1] = ch.out[:, :n].cpu().numpy()          # one D2H per chunk
        del ch                                            # before the next chunk is allocated
    return out


def _labels(ests, dec):
    """Rows of predict(): the decision rows, or for classifiers their labels through each model's binarizer."""
    if isinstance(ests[0], ClassifierMixin):
        return [e.label_binarizer_.inverse_transform(dec[b] > 0) for b, e in enumerate(ests)]
    return list(dec)


def predict_many(estimators, X):
    """Predictions of many fitted estimators on one design matrix: [n_models, n_samples], row b equal to
    estimators[b].predict(X) (classifiers: labels through each model's own label_binarizer_; when the models' label
    types differ, an object array).  The estimators are those decision_function_many accepts."""
    ests = list(estimators)
    if not ests:
        return _decision(ests, X, "predict_many")
    rows = _labels(ests, _decision(ests, X, "predict_many"))
    if len({r.dtype for r in rows}) == 1:
        return np.stack(rows)
    out = np.empty((len(rows), len(rows[0])), dtype=object)
    for b, r in enumerate(rows):
        out[b] = r
    return out


def _check_targets(ests, y, n, what):
    ys = _targets(y, len(ests), what)
    for b, yb in enumerate(ys):
        if len(yb) != n:
            raise ValueError(f"{what}: target {b} has {len(yb)} samples and X has {n}")
    return ys


def score_many(estimators, X, y):
    """Scores of many fitted estimators on one design matrix: ndarray [n_models], entry b equal to
    estimators[b].score(X, y_b) -- R^2 for regressors, accuracy for classifiers -- computed on the host from
    predict_many.  y: one target array for every model, or a sequence of one per estimator (one-vs-rest)."""
    ests = list(estimators)
    if not ests:
        return np.zeros(0)
    fm, Xc, shape = _prepare(ests, X, "score_many")
    ys = _check_targets(ests, y, Xc.shape[0], "score_many")
    rows = _labels(ests, _device_decision(ests, fm, Xc, shape, "score_many"))
    metric = accuracy_score if isinstance(ests[0], ClassifierMixin) else r2_score
    return np.array([float(metric(yb, r)) for yb, r in zip(ys, rows)])


def objective_many(estimators, X, y):
    """objective(est, X, y_b) of many fitted estimators on one design matrix: a list of dicts (loss, l2_w, l2_P,
    omega, total), entry b equal to sparsepoly_b200.objective(estimators[b], X, y_b) key by key, bit for bit.  y: one
    target array for every model, or a sequence of one per estimator.  Each reduction is one launch pair over all
    models of a chunk (Omega: at most two partial launches, one per fold kind, per order); the estimators are those
    decision_function_many accepts."""
    ests = list(estimators)
    if not ests:
        return []
    what = "objective_many"
    fm, Xc, shape = _prepare(ests, X, what)
    n = Xc.shape[0]
    ys = _check_targets(ests, y, n, what)
    n_orders, k, d = shape if fm else (1,) + shape
    results = []
    for b0, b1, ch in _run_chunks(ests, Xc, fm, shape, what, objective=True):
        results += _chunk_objective(ests[b0:b1], ys[b0:b1], ch, fm, n, n_orders, k, d)
        del ch                                            # before the next chunk is allocated
    return results


def _chunk_objective(chunk, ys, ch, fm, n, n_orders, k, d):
    first = chunk[0]
    B, dev = len(chunk), ch.out.device
    y_dev = torch.zeros((B, max(n, 1)), dtype=_f64)
    if n > 0:
        y_dev[:, :n] = torch.from_numpy(np.stack([_objective._targets(e, yb) for e, yb in zip(chunk, ys)]))
    y_dev = y_dev.to(dev)
    parts = torch.zeros((4, B), dtype=_f64, device=dev)          # loss, l2_w, l2_P, omega
    sum_work = torch.empty(B * solvers.sum_work_doubles(), dtype=_f64, device=dev)
    loss_tab = (_lib.SpLossEntry * B)()
    for b, e in enumerate(chunk):
        loss_tab[b] = _lib.SpLossEntry(y_pred=ch.out[b].data_ptr(), y=y_dev[b].data_ptr(),
                                       loss=_lib.LOSS_IDS[e.loss], out=parts[0, b].data_ptr())
    solvers.loss_sum_multi(loss_tab, n, sum_work)
    if fm and first.fit_linear:
        w_tab = (_lib.SpSqnormEntry * B)()
        for b in range(B):
            w_tab[b] = _lib.SpSqnormEntry(v=ch.w[b].data_ptr(), out=parts[1, b].data_ptr())
        solvers.sqnorm_multi(w_tab, d, sum_work)
    reg_work = torch.empty(B * solvers.reg_eval_work_doubles(d, k), dtype=_f64, device=dev)
    per_order = torch.empty((2, B), dtype=_f64, device=dev)
    for o in range(n_orders):                       # l2_P and omega: 0 + order 0 + order 1 ..., as objective()
        sq_tab, reg_tab = (_lib.SpSqnormEntry * B)(), (_lib.SpRegEntry * B)()
        for b, e in enumerate(chunk):
            P = ch.P_dk[b, o].data_ptr()
            sq_tab[b] = _lib.SpSqnormEntry(v=P, out=per_order[0, b].data_ptr())
            reg_tab[b] = _lib.SpRegEntry(P_dk=P, reg=_lib.REG_IDS[e.regularizer], out=per_order[1, b].data_ptr())
        solvers.sqnorm_multi(sq_tab, d * k, sum_work)
        solvers.reg_eval_multi(reg_tab, d, k, first.degree - o if fm else -1, reg_work)
        parts[2:] += per_order
    host = parts.cpu().numpy()                      # one D2H per chunk
    results = []
    for b, e in enumerate(chunk):
        scale = n if e.mean else 1
        alpha = e.alpha * scale if fm else 0.0
        beta, gamma = e.beta * scale, e.gamma * scale
        out = dict(loss=float(host[0, b]), l2_w=float(host[1, b]), l2_P=float(host[2, b]), omega=float(host[3, b]))
        out["total"] = out["loss"] + 0.5 * alpha * out["l2_w"] + 0.5 * beta * out["l2_P"] + gamma * out["omega"]
        results.append(out)
    return results
