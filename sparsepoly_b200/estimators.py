"""sklearn-style estimators with the reference's public surface, fitted on the B200 backend.

Drop-in for reference sparsepoly/{base,sparse_factorization_machines,sparse_all_subsets}.py:
same class names, constructor parameters / defaults, fitted attributes (P_, w_, lams_,
n_iter_, it_, label_binarizer_), warnings and verbose strings.  What changed is below the
boundary: the Dataset / Loss / Regularizer jitclasses and the @njit epoch functions are
replaced by device buffers and calls into libsparsepoly_b200.so (solvers.py).

Differences from the reference that are deliberate and documented in DESIGN.md:
  * unsupported solver x regularizer x degree combinations raise ValueError up front (the
    reference fails with a numba TypingError when the epoch function is compiled);
  * `callback(self)` sees the CURRENT P_ / w_ for every solver (the reference exposes a stale
    pre-fit copy for pbcd / psgd, sparse_factorization_machines.py:285 vs :352);
  * the initial predictions use the DP kernel instead of the power-sum identities
    (kernels.py:91-114): same value up to ~1e-16 relative rounding.
"""
import warnings
from abc import ABCMeta, abstractmethod

import numpy as np
import torch
from sklearn.base import BaseEstimator, ClassifierMixin, RegressorMixin
from sklearn.exceptions import NotFittedError
from sklearn.preprocessing import LabelBinarizer, add_dummy_feature
from sklearn.utils import check_random_state
from sklearn.utils.multiclass import type_of_target
from sklearn.utils.validation import check_consistent_length, column_or_1d

from . import _lib, cd, solvers
from .dataset import DeviceCSR, DeviceDataset, _use_device, check_X, check_X_y, host_y
from .distributed import active_group, broadcast_arrays, global_sum

REGRESSION_LOSSES = ("squared",)
CLASSIFICATION_LOSSES = ("squared", "squared_hinge", "logistic")
FM_REGULARIZERS = ("squaredl12", "squaredl21", "l1", "l21", "omegati", "omegacs")
ALL_SUBSETS_REGULARIZERS = ("l1", "l21", "omegacs", "omegati")
LEARNING_RATE = _lib.LEARNING_RATE

# which regularizers implement which solver protocol (reference README.md:25-31 and the
# methods each jitclass defines, regularizer/*.py)
_SOLVER_REGS = {
    "pcd": ("l1", "squaredl12", "omegati"),
    "pbcd": ("l1", "l21", "squaredl21", "omegacs"),
    "psgd": ("l1", "l21", "squaredl12", "squaredl21"),
}

_f64 = torch.float64


def _process_group():
    """Sharded psgd is opt-in (distributed.enable_sharding); an initialised torch.distributed alone
    changes nothing."""
    return active_group()


class _SparsePolyBase(BaseEstimator, metaclass=ABCMeta):
    """Shared validation (reference base.py:17-34)."""

    def _get_loss(self, loss):
        if loss not in self._LOSSES:
            losses_str = '", "'.join(self._LOSSES)
            raise ValueError(f"Loss function {loss} not supported. The available options are:"
                             f' "{losses_str}".')
        return loss

    def _get_regularizer(self, regularizer):
        if regularizer not in self._REGULARIZERS:
            regularizers_str = '", "'.join(self._REGULARIZERS)
            raise ValueError(f"Regularizer {regularizer} not supported. The available options are:"
                             f' "{regularizers_str}".')
        return regularizer

    def _check_combination(self, solver, regularizer, degree):
        if solver not in _SOLVER_REGS:
            raise ValueError(f"Solver {solver} is not supported.")
        if regularizer not in _SOLVER_REGS[solver]:
            raise ValueError(f"Regularizer {regularizer} cannot be used with solver {solver}; "
                             f"{solver} supports: {', '.join(_SOLVER_REGS[solver])}.")
        if solver == "pcd" and regularizer == "squaredl12" and degree > 2:
            raise ValueError("SquaredL12 supports only degree=2.")       # squaredl12.py:25-26
        if solver == "pbcd" and regularizer == "squaredl21" and degree != 2:
            raise ValueError("SquaredL21 supports only degree=2.")       # squaredl21.py:28-29

    def _init_lambdas(self, rng):
        if not (self.warm_start and hasattr(self, "lams_")):
            if self.init_lambdas == "ones":
                self.lams_ = np.ones(self.n_components)
            elif self.init_lambdas == "random_signs":
                self.lams_ = np.sign(rng.randn(self.n_components))
            else:
                raise ValueError("Lambdas must be initialized as ones (init_lambdas='ones') or as "
                                 "random +/- 1 (init_lambdas='random_signs').")

    def __getstate__(self):
        # device handles (ctypes structs with pointers, CUDA tensors) are per-fit scratch, not model state:
        # a fitted estimator pickles / deep-copies like the reference's (P_, w_, lams_, ... are numpy)
        state = dict(self.__dict__)
        for key in ("_dev_state", "_psgd_stream"):
            state.pop(key, None)
        return state

    def _cd_setup(self, X, y, rng, dev):
        """pcd / pbcd: move everything to the device and return (epoch, sync), see cd.setup."""
        return cd.setup(self, X, y, rng, dev)

    def _after_epoch(self, it, value, what, sync):
        """callback / verbose handling shared by the epoch loops; True = stop."""
        if (self.callback is not None) and it % self.n_calls == 0:
            sync()
            if self.callback(self) is not None:
                return True
        if self.verbose:
            print(what.format(it + 1, value))
        return False


class SparsePolyRegressorMixin(RegressorMixin):
    """reference base.py:37-65."""
    _LOSSES = REGRESSION_LOSSES

    def _check_X_y(self, X, y):
        X, y = check_X_y(X, y, accept_sparse=True, multi_output=False, dtype=np.double,
                         y_numeric=True)
        return X, y.astype(np.double).ravel()

    def _partial_fit_X_y(self, X, y, classes):
        """X, y of one partial_fit call (classes is the classifier's; ignored here) and no label binarizer."""
        X, y = self._check_X_y(X, y)
        return X, y, None

    def predict(self, X):
        """Predict regression output for the samples in X ([n_samples] array)."""
        return self._predict(X)


class SparsePolyClassifierMixin(ClassifierMixin):
    """reference base.py:68-142."""
    _LOSSES = CLASSIFICATION_LOSSES

    def decision_function(self, X):
        """Model output before thresholding ([n_samples] array)."""
        return self._predict(X)

    def predict(self, X):
        """Predicted class labels for the samples in X."""
        y_pred = self.decision_function(X) > 0
        return self.label_binarizer_.inverse_transform(y_pred)

    def predict_proba(self, X):
        """Probability of the positive class; only available if loss='logistic'."""
        if self.loss == "logistic":
            return 1 / (1 + np.exp(-self.decision_function(X)))
        raise ValueError("Probability estimates only available for loss='logistic'. You may use "
                         "probability calibration methods from scikit-learn instead.")

    @staticmethod
    def _binary_labels(y):
        """(classes, y in {-1, +1}) of a 1-D numeric label array with exactly two integer-valued classes, else
        None.  Same result as type_of_target + LabelBinarizer(pos_label=1, neg_label=-1) below, without their
        sorts: a few streaming passes (0.03 s instead of 0.4 s at 6 M labels)."""
        if not isinstance(y, np.ndarray) or y.ndim != 1 or y.size == 0 or y.dtype.kind not in "fiu":
            return None
        lo, hi = y.min(), y.max()
        if not (np.isfinite(lo) and np.isfinite(hi) and lo < hi) or lo != np.floor(lo) or hi != np.floor(hi):
            return None
        is_hi = y == hi
        if not np.all(is_hi | (y == lo)):
            return None
        return np.array([lo, hi], dtype=y.dtype), np.where(is_hi, 1.0, -1.0)

    def _check_X_y(self, X, y):
        y = host_y(y)
        fast = self._binary_labels(y)
        if fast is not None:
            X = check_X(X, dtype=np.double, accept_sparse=True)
            check_consistent_length(X, y)
            lb = LabelBinarizer(pos_label=1, neg_label=-1)
            lb.classes_, lb.y_type_, lb.sparse_input_ = fast[0], "binary", False
            self.label_binarizer_ = lb
            return X, fast[1]
        is_2d = hasattr(y, "shape") and len(y.shape) > 1 and y.shape[1] >= 2
        if is_2d or type_of_target(y) != "binary":
            raise TypeError("Only binary targets supported. For training multiclass or multilabel "
                            "models, you may use the OneVsRest or OneVsAll metaestimators in "
                            "scikit-learn.")
        X, Y = check_X_y(X, y, dtype=np.double, accept_sparse=True, multi_output=False)
        self.label_binarizer_ = LabelBinarizer(pos_label=1, neg_label=-1)
        y = self.label_binarizer_.fit_transform(Y).ravel().astype(np.double)
        return X, y

    def _partial_fit_X_y(self, X, y, classes):
        """X, y in {-1, +1} of one partial_fit call, and the label binarizer of `classes` when the estimator has
        none yet (the first call of a stream: classes is required there and ignored later, as in scikit-learn).
        A chunk may hold one class only; labels map to +-1 as LabelBinarizer(pos_label=1, neg_label=-1) maps
        them in fit."""
        lb = getattr(self, "label_binarizer_", None)
        new = None
        if lb is not None and classes is not None and not np.array_equal(np.unique(classes), lb.classes_):
            raise ValueError(f"classes={list(classes)!r} differs from the classes the model was fitted with "
                             f"({lb.classes_.tolist()}).")
        if lb is None:
            if classes is None:
                raise ValueError("classes must be passed on the first call to partial_fit.")
            classes = np.asarray(classes)
            if classes.ndim != 1 or classes.size != 2 or np.unique(classes).size != 2:
                raise ValueError(f"classes must hold exactly two distinct labels, got {classes!r}.")
            lb = new = LabelBinarizer(pos_label=1, neg_label=-1).fit(classes)
        X = check_X(X, dtype=np.double, accept_sparse=True)
        y = column_or_1d(host_y(y))
        check_consistent_length(X, y)
        known = np.isin(y, lb.classes_)
        if not np.all(known):
            raise ValueError(f"y contains labels that are not in classes {lb.classes_.tolist()}: "
                             f"{np.unique(y[~known])[:5].tolist()}")
        return X, np.where(y == lb.classes_[1], 1.0, -1.0), new


# =============================================================================================
# Factorization machines
# =============================================================================================
class _BaseSparseFactorizationMachine(_SparsePolyBase, metaclass=ABCMeta):
    _REGULARIZERS = FM_REGULARIZERS

    @abstractmethod
    def __init__(self, degree=2, loss="squared", n_components=2, solver="pcd",
                 regularizer="squaredl12", alpha=1, beta=1, gamma=1, mean=False, tol=1e-6,
                 fit_lower="explicit", fit_linear=True, warm_start=False, init_lambdas="ones",
                 max_iter=100, shuffle=False, batch_size="auto", eta0=1.0, learning_rate="optimal",
                 power_t=1.0, n_iter_no_change=5, verbose=False, callback=None, n_calls=10,
                 random_state=None):
        self.degree = degree
        self.loss = loss
        self.n_components = n_components
        self.solver = solver
        self.regularizer = regularizer
        self.alpha = alpha
        self.beta = beta
        self.gamma = gamma
        self.mean = mean
        self.tol = tol
        self.fit_lower = fit_lower
        self.fit_linear = fit_linear
        self.warm_start = warm_start
        self.init_lambdas = init_lambdas
        self.max_iter = max_iter
        self.shuffle = shuffle
        self.batch_size = batch_size
        self.eta0 = eta0
        self.learning_rate = learning_rate
        self.power_t = power_t
        self.n_iter_no_change = n_iter_no_change
        self.verbose = verbose
        self.callback = callback
        self.n_calls = n_calls
        self.random_state = random_state

    # ---------------------------------------------------------------- helpers
    def _augment(self, X):
        # one dummy all-ones column per missing lower order (sparse_factorization_machines.py:86-92)
        if self.fit_lower == "augment":
            k = 2 if self.fit_linear else 1
            if isinstance(X, DeviceCSR):
                return X.augment(max(0, self.degree - k))
            for _ in range(self.degree - k):
                X = add_dummy_feature(X, value=1)
        return X

    def _scaled(self, n_samples):
        if self.mean:
            return self.alpha * n_samples, self.beta * n_samples, self.gamma * n_samples
        return self.alpha, self.beta, self.gamma

    def _output_orders(self):
        """(order index, degree) pairs that enter the prediction (quirk kept: explicit lower
        orders are only added for degree == 3, sparse_factorization_machines.py:445-449)."""
        orders = [(0, self.degree)]
        if self.fit_lower == "explicit" and self.degree == 3:
            orders.append((1, 2))
        return orders

    def _device_output(self, ds, P_kd_orders, w_dev, lams_dev, out, stride):
        """_get_output on device: writes the model output into out[::stride]."""
        first = True
        for o, deg in self._output_orders():
            P_dk = solvers.transpose(P_kd_orders[o])
            solvers.poly_predict(ds, P_dk, lams_dev, deg, w=w_dev if (first and self.fit_linear) else None,
                                 out=out, out_stride=stride, accumulate=not first)
            first = False
        return out

    def _init_coefs(self, n_features, rng):
        """w_, P_ and lams_ at the start of fit (kept under warm_start); draws P_ then the lambdas from rng."""
        if not (self.warm_start and hasattr(self, "w_")):
            self.w_ = np.zeros(n_features, dtype=np.double)
        n_orders = self.degree - 1 if self.fit_lower == "explicit" else 1
        if not (self.warm_start and hasattr(self, "P_")):
            self.P_ = 0.01 * rng.randn(n_orders, self.n_components, n_features)
        self._init_lambdas(rng)
        if np.unique(np.abs(self.lams_)) != np.array([1.0]):
            raise ValueError("Lambdas must be +1 or -1.")

    _pcd_setup = _pbcd_setup = _SparsePolyBase._cd_setup

    # ---------------------------------------------------------------- psgd
    def _start_upload(self, X, dev):
        """psgd: X moves to the device on a helper thread while fit() draws the initial P on this one (numpy's
        generators and the copies both release the GIL); _psgd_setup joins it."""
        import threading
        box = {}
        planned = self.regularizer in solvers.PLANNED_REGS

        def work():
            try:
                torch.cuda.set_device(dev)
                _use_device(dev)
                box["ds"] = DeviceDataset(X, need_csr=True, need_csc=False, device=dev, hot_features=not planned)
            except BaseException as e:          # re-raised by the joining thread
                box["error"] = e
        th = threading.Thread(target=work, daemon=True)
        th.start()
        return th, box

    def _psgd_settings(self):
        """(learning-rate id, process group, world, rank) of a psgd fit."""
        if self.learning_rate not in LEARNING_RATE:
            raise ValueError(f"learning_rate {self.learning_rate} is not supported."
                             f" Choose from {LEARNING_RATE}.")
        group = _process_group()
        world, rank = 1, 0
        if group is not None:
            import torch.distributed as dist
            world, rank = dist.get_world_size(group), dist.get_rank(group)
        return LEARNING_RATE[self.learning_rate], group, world, rank

    def _psgd_model(self, dev, batch_size, learning_rate, group=None, world=1, rank=0):
        """The model half of psgd, which outlives a pass over the rows: P_ / w_ / lams_ on the device, the loss
        accumulator and the dense-gradient path's buffers.  The planned path's context joins it with the first
        plan (_psgd_bind)."""
        d, k = self.P_.shape[2], self.n_components
        P = solvers.transpose_batch(torch.from_numpy(np.ascontiguousarray(self.P_)).to(dev))   # [n_orders, d, k]
        m = dict(planned=self.regularizer in solvers.PLANNED_REGS, learning_rate=learning_rate, group=group,
                 world=world, rank=rank, batch_size=batch_size, b_loc=max(1, batch_size // world), P=P,
                 w=torch.from_numpy(np.ascontiguousarray(self.w_)).to(dev),
                 lams=torch.from_numpy(np.ascontiguousarray(self.lams_, dtype=np.float64)).to(dev),
                 loss=torch.zeros(1, dtype=_f64, device=dev), model_current=True, ctx=None)
        if not m["planned"]:
            m.update(grad_P=torch.zeros_like(P), grad_w=torch.zeros(d, dtype=_f64, device=dev),
                     work=solvers.prox_work(d, k, dev))
        return m

    @staticmethod
    def _psgd_data(ds, y, order, dev):
        """The data half of a psgd pass: the rows, their targets and the order they are visited in (the planned
        path adds the batch-CSC plan of that order, _psgd_plan)."""
        return dict(ds=ds, n=ds.n_samples, order=order, y=torch.from_numpy(y).to(dev),
                    idx=torch.from_numpy(order).to(dev), plan=None)

    @staticmethod
    def _psgd_plan(m, data):
        from .psgd_plan import PsgdPlan
        return PsgdPlan(data["ds"].csr, data["idx"], data["ds"].n_features, m["b_loc"], world=m["world"],
                        rank=m["rank"], group=m["group"])

    def _psgd_bind(self, m, plan, inbox_cap=None):
        """Planned path: the context runs on `plan`.  The first plan creates it (model loaded, frame and selection
        state reset); later plans (reshuffles, further partial_fit chunks) only grow its plan-sized scratch."""
        if m["ctx"] is not None:
            m["ctx"].rebind(plan)
            return
        from .psgd_plan import PsgdContext
        ctx = PsgdContext(plan, m["P"].shape[0], self.n_components, self.degree, self.regularizer, self.loss,
                          self.fit_linear, m["lams"], group=m["group"], inbox_cap=inbox_cap)
        ctx.load_model(m["P"], m["w"])
        solvers.psgd_planned_begin(ctx)
        m["ctx"] = ctx

    def _psgd_pass(self, m, data, n_glob, read_back=True):
        """One psgd.psgd_epoch (sparse_factorization_machines.py:123-150) over the rows of `data` in its order:
        advances it_ and returns the mean loss (None with read_back=False).  l1 / squaredl12 run the planned path
        (psgd_plan.cu: gather passes over a batch-CSC plan, touched rows only, sharded over peer memory); l21 /
        squaredl21 the dense-gradient path (psgd.cu)."""
        ctx, loss = m["ctx"], m["loss"]
        loss.zero_()
        if m["planned"]:
            self.it_ = solvers.psgd_planned_run(ctx, data["ds"], data["plan"], data["y"], data["idx"], self.alpha,
                                                self.beta, self.gamma, self.eta0, m["learning_rate"], self.power_t,
                                                self.it_)
            # (the run folds the lazy scales back into the storage after any minibatch that takes them out of
            # (1e-100, 1e100); sync() materialises the frame the pass leaves)
            solvers.psgd_planned_end(ctx, data["n"], loss, False)
            m["model_current"] = False
        else:
            self.it_ = solvers.psgd_epoch(data["ds"], data["y"], m["P"], m["w"], m["lams"], self.degree, self.alpha,
                                          self.beta, self.gamma, self.regularizer, self.loss, m["grad_P"],
                                          m["grad_w"], data["idx"], self.fit_linear, self.eta0, m["learning_rate"],
                                          self.power_t, m["batch_size"], self.it_, loss, m["work"], m["group"])
        if not read_back:
            return None
        sum_loss = loss.item()
        if m["planned"]:
            ctx.check_peers()
        if m["group"] is not None:
            sum_loss = global_sum([sum_loss], m["group"])[0]
        return sum_loss / n_glob

    def _psgd_setup(self, X, y, rng, dev, upload=None):
        """Move everything to the device and return (epoch, sync, close): epoch() is one _psgd_pass over all of X,
        reshuffled first with shuffle=True."""
        n, d = X.shape
        learning_rate, group, world, rank = self._psgd_settings()
        if group is not None:
            # replicas must start identical whatever each rank's random_state drew, and shards must be equal
            it_arr = np.array([float(self.it_)])
            broadcast_arrays([self.P_, self.w_, self.lams_, it_arr], group)
            self.it_ = int(it_arr[0])
            sizes = global_sum([float(n), float(n) ** 2], group)
            if abs(sizes[1] * world - sizes[0] ** 2) > 0.5:
                raise ValueError("sharded psgd needs the same number of samples on every rank")
        planned = self.regularizer in solvers.PLANNED_REGS
        import os
        import time
        timing = os.environ.get("SPARSEPOLY_B200_TIMING") == "1"

        def _tick():
            if timing:
                torch.cuda.synchronize()
            return time.perf_counter()
        t0 = _tick()
        if upload is not None:
            upload[0].join()
            if "error" in upload[1]:
                raise upload[1]["error"]
            ds = upload[1]["ds"]
        else:
            ds = DeviceDataset(X, need_csr=True, need_csc=False, device=dev, hot_features=not planned)
        t1 = _tick()
        self._h2d_bytes = ds.h2d_bytes + y.nbytes + self.P_.nbytes + self.w_.nbytes
        n_glob, nnz_glob = (global_sum([n, ds.nnz], group) if group is not None else (n, ds.nnz))
        if self.batch_size == "auto":
            batch_size = int(n_glob * d / nnz_glob)                          # :101-102
        else:
            batch_size = self.batch_size
        batch_size = max(int(batch_size), 1)
        data = self._psgd_data(ds, y, np.arange(n, dtype=np.int32), dev)
        m = self._psgd_model(dev, batch_size, learning_rate, group, world, rank)
        if planned:
            t2 = _tick()
            data["plan"] = plan = self._psgd_plan(m, data)
            t3 = _tick()
            self._psgd_bind(m, plan, inbox_cap=(min(plan.d_rows, m["b_loc"] * int(ds.max_row_nnz()))
                                                if self.shuffle else None))     # (shuffle=True: bound for any order)
            self._psgd_stats = {"plan_bytes": plan.nbytes(), "minibatches": plan.n_minibatches,
                                "columns_per_minibatch": plan.n_cols / max(plan.n_minibatches, 1),
                                "batch_size": batch_size, "batch_local": m["b_loc"], "world": world,
                                "setup_seconds": {"upload_X": t1 - t0, "upload_model": t2 - t1, "plan": t3 - t2,
                                                  "context": _tick() - t3, "synchronised": timing}}
        else:
            self._psgd_stats = {"batch_size": batch_size, "world": world}

        def sync():
            P, w = m["P"], m["w"]
            if planned:
                if not m["model_current"]:
                    solvers.psgd_planned_end(m["ctx"], 0, None, True)
                    m["model_current"] = True
                m["ctx"].store_model(P, w)
            self.P_[...] = solvers.transpose_batch(P).cpu().numpy()
            self.w_[...] = w.cpu().numpy()

        def epoch(read_back=True):
            if self.shuffle:
                rng.shuffle(data["order"])
                data["idx"].copy_(torch.from_numpy(data["order"]))
                if planned:
                    data["plan"] = self._psgd_plan(m, data)
                    self._psgd_bind(m, data["plan"])
            return self._psgd_pass(m, data, n_glob, read_back)

        def close():
            if planned:
                if self.regularizer == "squaredl12":
                    self._psgd_stats["selection"] = solvers.psgd_planned_solver_stats(m["ctx"])
                m["ctx"].close()

        return epoch, sync, close

    def _fit_psgd(self, X, y, rng, dev, upload=None):
        """sparse_factorization_machines.py:94-173 (epoch loop, plateau stopping rule :157-170)."""
        epoch_fn, sync, close = self._psgd_setup(X, y, rng, dev, upload)
        converged, epoch = False, 0
        no_improvement_count, best_loss = 0, np.inf
        try:
            for epoch in range(self.max_iter):
                sum_loss = epoch_fn()
                if self._after_epoch(epoch, sum_loss, "Epoch {} loss {}", sync):
                    break
                if sum_loss > (best_loss - self.tol):
                    no_improvement_count += 1
                else:
                    no_improvement_count = 0
                if sum_loss < best_loss:
                    best_loss = sum_loss
                if no_improvement_count >= self.n_iter_no_change:
                    if self.verbose:
                        print(f"Converged at iteration {epoch+1}")
                    converged = True
                    break
            sync()
        finally:
            close()
        return converged, epoch

    # ---------------------------------------------------------------- public
    def fit(self, X, y):
        """Fit the factorization machine to (X, y) on the current CUDA device; returns self."""
        X, y = self._check_X_y(X, y)
        X = self._augment(X)
        n_features = X.shape[1]
        rng = check_random_state(self.random_state)
        self._get_loss(self.loss)
        self._get_regularizer(self.regularizer)
        if self.solver not in ("pcd", "pbcd", "psgd"):
            raise ValueError(f"Solver {self.solver} is not supported.")
        self._check_combination(self.solver, self.regularizer, self.degree)
        self._end_stream()
        dev = _use_device()
        upload = self._start_upload(X, dev) if self.solver == "psgd" and not isinstance(X, DeviceCSR) else None

        self._init_coefs(n_features, rng)

        y = np.ascontiguousarray(y, dtype=np.float64)
        if self.solver == "psgd":
            if not (self.warm_start and hasattr(self, "it_")):
                self.it_ = 1
            converged, self.n_iter_ = self._fit_psgd(X, y, rng, dev, upload)
            if not converged:
                warnings.warn("Objective did not converge. Increase max_iter.")
        else:
            epoch, sync = self._cd_setup(X, y, rng, dev)
            cd.stopping_loop([self], [sync], lambda active: [epoch()])
        return self

    def partial_fit(self, X, y, classes=None):
        """One pass of psgd over the rows of (X, y), continuing the model and the optimiser state of the earlier
        calls: trains on data too large for the device, streamed from the host in chunks of rows.  Returns self.

        The rows are cut into minibatches of batch_size from the call's first row (the last one may be short;
        nothing is carried to the next call); it_ continues across calls and n_iter_ counts them.  Chunks of a
        multiple of batch_size rows, passed in order E times with shuffle=False, give the model of
        fit(max_iter=E) on their concatenation.  P_ / w_ are current after every call.  The first call starts from
        the drawn initial model, or from the fitted one if there is one; the classifier's first call needs
        `classes` (the two labels).  fit() afterwards starts over.  solver='psgd' on one GPU only."""
        import time
        t0 = time.perf_counter()
        if self.solver != "psgd":
            raise ValueError(f"partial_fit is implemented for solver='psgd' only (got solver={self.solver!r}).")
        self._get_loss(self.loss)
        self._get_regularizer(self.regularizer)
        self._check_combination(self.solver, self.regularizer, self.degree)
        learning_rate, group, _, _ = self._psgd_settings()
        if group is not None:
            raise ValueError("partial_fit runs psgd on one GPU; sharded psgd (distributed.enable_sharding) is not "
                             "supported by it.")
        X, y, label_binarizer = self._partial_fit_X_y(X, y, classes)
        X = self._augment(X)
        n, n_features = X.shape
        if hasattr(self, "P_") and self.P_.shape[-1] != n_features:
            raise ValueError(f"X has {n_features} features (after fit_lower), but the model has "
                             f"{self.P_.shape[-1]}.")
        n_orders = self.degree - 1 if self.fit_lower == "explicit" else 1
        if hasattr(self, "P_") and self.P_.shape[:2] != (n_orders, self.n_components):
            raise ValueError(f"degree / fit_lower / n_components ask for {n_orders} order(s) of {self.n_components} "
                             f"components, but the model has P_ of shape {self.P_.shape}; fit() starts a new model.")
        m = getattr(self, "_psgd_stream", None)
        if m is not None and m["config"] != self._stream_config():
            raise ValueError("degree / n_components / regularizer / loss / fit_lower / fit_linear changed since the "
                             "stream started; fit() starts a new model.")
        t1 = time.perf_counter()
        dev = _use_device()
        before = dict(self.__dict__) if m is None else None
        try:
            mean_loss = self._stream_call(X, y, label_binarizer, learning_rate, dev, m, t0, t1)
        except BaseException:
            if before is not None:                  # a failed first call leaves the estimator as it was
                new = self.__dict__.get("_psgd_stream")
                if new is not None and new["ctx"] is not None:
                    new["ctx"].close()
                self.__dict__.clear()
                self.__dict__.update(before)
            raise
        if self.verbose:
            print(f"Call {self.n_iter_} loss {mean_loss}")
        return self

    def _stream_config(self):
        return (self.degree, self.n_components, self.regularizer, self.loss, self.fit_lower, self.fit_linear)

    def _stream_call(self, X, y, label_binarizer, learning_rate, dev, m, t0, t1):
        """The device part of partial_fit (m: the stream's model half, None on the first call of a process);
        returns the call's mean loss and leaves the phase times in _partial_fit_stats."""
        import time
        n, n_features = X.shape
        if label_binarizer is not None:
            self.label_binarizer_ = label_binarizer
        if m is None and not hasattr(self, "batch_size_"):     # a new stream (an unpickled one goes on as it was)
            self._stream_rng = check_random_state(self.random_state)
            self.n_iter_ = 0
            if not hasattr(self, "P_"):
                self._init_coefs(n_features, self._stream_rng)
            self.it_ = getattr(self, "it_", 1)
        t2 = time.perf_counter()
        planned = self.regularizer in solvers.PLANNED_REGS
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
        ev[0].record()
        ds = DeviceDataset(X, need_csr=True, need_csc=False, device=dev, hot_features=not planned)
        if not hasattr(self, "batch_size_"):
            self.batch_size_ = max(int(n * n_features / ds.nnz) if self.batch_size == "auto"    # :101-102
                                   else int(self.batch_size), 1)
        order = np.arange(n, dtype=np.int32)
        if self.shuffle:
            self._stream_rng.shuffle(order)
        data = self._psgd_data(ds, np.ascontiguousarray(y, dtype=np.float64), order, dev)
        ev[1].record()
        if m is None:
            m = self._psgd_model(dev, self.batch_size_, learning_rate)
            m["config"] = self._stream_config()
        ev[2].record()
        if planned:
            data["plan"] = self._psgd_plan(m, data)
            self._psgd_bind(m, data["plan"])
        ev[3].record()
        self._psgd_stream = m
        mean_loss = self._psgd_pass(m, data, n)
        ev[4].record()
        t3 = time.perf_counter()
        self._psgd_read(m)
        self.n_iter_ += 1
        sec = lambda i: ev[i].elapsed_time(ev[i + 1]) / 1e3          # noqa: E731
        self._partial_fit_stats = {"rows": n, "validate_s": t1 - t0, "h2d_s": sec(0), "model_s": t2 - t1 + sec(1),
                                   "plan_s": sec(2), "minibatches_s": sec(3), "readout_s": time.perf_counter() - t3}
        return mean_loss

    def _psgd_read(self, m):
        """P_ / w_ of the stream's model, the device state left as it is: the planned path reads the lazy frame
        (sp_psgd_plan_read) instead of materialising it, which would change the rounding of the calls to come."""
        P = m["P"]
        n_orders, d, k = P.shape
        if m["planned"]:
            P_out = torch.empty((n_orders, k, d), dtype=_f64, device=P.device)
            w_out = torch.empty(d, dtype=_f64, device=P.device)
            solvers.psgd_planned_read(m["ctx"], P_out, w_out)
        else:
            P_out, w_out = solvers.transpose_batch(P), m["w"]
        self.P_, self.w_ = P_out.cpu().numpy(), w_out.cpu().numpy()

    def _end_stream(self):
        """fit starts over: the device state of a partial_fit stream is released and its attributes dropped."""
        m = self.__dict__.pop("_psgd_stream", None)
        if m is not None and m["ctx"] is not None:
            m["ctx"].close()
        for key in ("_stream_rng", "batch_size_", "_partial_fit_stats"):
            self.__dict__.pop(key, None)

    def _get_output(self, X):
        dev = _use_device()
        ds = DeviceDataset(X, need_csr=True, need_csc=False, device=dev)
        P = torch.from_numpy(np.ascontiguousarray(self.P_)).to(dev)
        w = torch.from_numpy(np.ascontiguousarray(self.w_)).to(dev)
        lams = torch.from_numpy(np.ascontiguousarray(self.lams_, dtype=np.float64)).to(dev)
        out = torch.zeros(ds.n_samples, dtype=_f64, device=dev)
        self._device_output(ds, P, w, lams, out, 1)
        return out.cpu().numpy()

    def _predict(self, X):
        if not hasattr(self, "P_"):
            raise NotFittedError("Estimator not fitted.")
        X = check_X(X, accept_sparse=["csr", "csc"], dtype=np.double)
        X = self._augment(X)
        return self._get_output(X)


class SparseFactorizationMachineRegressor(_BaseSparseFactorizationMachine, SparsePolyRegressorMixin):
    """Sparse factorization machine for regression (squared loss) on the B200 backend.

    Parameters, defaults, fitted attributes and semantics are those of the reference class of the
    same name (sparse_factorization_machines.py:461-685): degree-m ANOVA model
    y(x) = <w,x> + sum_orders sum_s lams_s * A^deg(P_[order,s], x) minimising
    sum_i loss + alpha/2 |w|^2 + beta/2 |P|^2 + gamma * Omega(P) with solver in
    {'pcd','pbcd','psgd'} and regularizer in {'squaredl12','squaredl21','omegati','omegacs',
    'l1','l21'}.  fit_lower in {'explicit','augment',None}; see the reference docstring for the
    meaning of every knob -- they are unchanged.

    Attributes: P_ [n_orders, n_components, n_features], w_ [n_features], lams_ [n_components],
    n_iter_, it_ (psgd).
    """
    _LOSSES = REGRESSION_LOSSES

    def __init__(self, degree=2, n_components=2, solver="pcd", regularizer="squaredl12", alpha=1,
                 beta=1, gamma=1, mean=False, tol=1e-6, fit_lower="explicit", fit_linear=True,
                 warm_start=False, init_lambdas="ones", max_iter=100, shuffle=False,
                 batch_size="auto", eta0=1.0, learning_rate="optimal", power_t=1.0,
                 n_iter_no_change=5, verbose=False, callback=None, n_calls=10, random_state=None):
        super().__init__(degree, "squared", n_components, solver, regularizer, alpha, beta, gamma,
                         mean, tol, fit_lower, fit_linear, warm_start, init_lambdas, max_iter,
                         shuffle, batch_size, eta0, learning_rate, power_t, n_iter_no_change,
                         verbose, callback, n_calls, random_state)


class SparseFactorizationMachineClassifier(_BaseSparseFactorizationMachine, SparsePolyClassifierMixin):
    """Sparse factorization machine for binary classification on the B200 backend.

    Same surface as the reference class (sparse_factorization_machines.py:688-920);
    loss in {'squared_hinge','logistic','squared'}; targets are binarised to {-1,+1}.
    """
    _LOSSES = CLASSIFICATION_LOSSES

    def __init__(self, degree=2, loss="squared_hinge", n_components=2, solver="pcd",
                 regularizer="squaredl12", alpha=1, beta=1, gamma=1, mean=False, tol=1e-6,
                 fit_lower="explicit", fit_linear=True, warm_start=False, init_lambdas="ones",
                 max_iter=100, shuffle=False, batch_size="auto", eta0=1.0, learning_rate="optimal",
                 power_t=1.0, n_iter_no_change=5, verbose=False, callback=None, n_calls=10,
                 random_state=None):
        super().__init__(degree, loss, n_components, solver, regularizer, alpha, beta, gamma, mean,
                         tol, fit_lower, fit_linear, warm_start, init_lambdas, max_iter, shuffle,
                         batch_size, eta0, learning_rate, power_t, n_iter_no_change, verbose,
                         callback, n_calls, random_state)


# =============================================================================================
# All-subsets models
# =============================================================================================
class _BaseSparseAllSubsets(_SparsePolyBase, metaclass=ABCMeta):
    _REGULARIZERS = ALL_SUBSETS_REGULARIZERS

    @abstractmethod
    def __init__(self, loss="squared", n_components=2, solver="pcd", beta=1, gamma=1, eta0=0.1,
                 mean=False, tol=1e-6, regularizer="omegati", warm_start=False, init_lambdas="ones",
                 max_iter=100, shuffle=False, verbose=False, callback=None, n_calls=10,
                 random_state=None):
        self.loss = loss
        self.n_components = n_components
        self.solver = solver
        self.beta = beta
        self.gamma = gamma
        self.eta0 = eta0
        self.mean = mean
        self.tol = tol
        self.regularizer = regularizer
        self.warm_start = warm_start
        self.init_lambdas = init_lambdas
        self.max_iter = max_iter
        self.shuffle = shuffle
        self.verbose = verbose
        self.callback = callback
        self.n_calls = n_calls
        self.random_state = random_state

    def fit(self, X, y):
        """Fit the all-subsets model to (X, y) on the current CUDA device; returns self."""
        X, y = self._check_X_y(X, y)
        d = X.shape[1]
        rng = check_random_state(self.random_state)
        self._get_loss(self.loss)
        self._get_regularizer(self.regularizer)
        if self.solver not in ("pcd", "pbcd"):
            raise ValueError(f"Solver {self.solver} is not supported.")
        self._check_combination(self.solver, self.regularizer, -1)
        dev = _use_device()
        self._init_coefs(d, rng)
        y = np.ascontiguousarray(y, dtype=np.float64)
        epoch, sync = self._setup(X, y, rng, dev)
        cd.stopping_loop([self], [sync], lambda active: [epoch()])
        return self

    def _init_coefs(self, n_features, rng):
        """P_ and lams_ at the start of fit (kept under warm_start); draws P_ then the lambdas from rng."""
        if not (self.warm_start and hasattr(self, "P_")):
            self.P_ = 0.01 * rng.randn(self.n_components, n_features)
        self._init_lambdas(rng)

    _setup = _SparsePolyBase._cd_setup

    def _get_output(self, X):
        dev = _use_device()
        ds = DeviceDataset(X, need_csr=True, need_csc=False, device=dev)
        P_dk = solvers.transpose(torch.from_numpy(np.ascontiguousarray(self.P_)).to(dev))
        lams = torch.from_numpy(np.ascontiguousarray(self.lams_, dtype=np.float64)).to(dev)
        return solvers.poly_predict(ds, P_dk, lams, -1).cpu().numpy()

    def _predict(self, X):
        if not hasattr(self, "P_"):
            raise NotFittedError("Estimator not fitted.")
        X = check_X(X, accept_sparse=["csr", "csc"], dtype=np.double)
        return self._get_output(X)


class SparseAllSubsetsRegressor(_BaseSparseAllSubsets, SparsePolyRegressorMixin):
    """Sparse all-subsets model y(x) = sum_s lams_s * prod_j (1 + P_[s,j] x_j) for regression.
    Same surface as the reference class (sparse_all_subsets.py:266-391)."""
    _LOSSES = REGRESSION_LOSSES

    def __init__(self, n_components=2, solver="pcd", beta=1, gamma=1, eta0=0.1, mean=False, tol=1e-6,
                 regularizer="omegati", warm_start=False, init_lambdas="ones", max_iter=100,
                 shuffle=False, verbose=False, callback=None, n_calls=10, random_state=None):
        super().__init__("squared", n_components, solver, beta, gamma, eta0, mean, tol, regularizer,
                         warm_start, init_lambdas, max_iter, shuffle, verbose, callback, n_calls,
                         random_state)


class SparseAllSubsetsClassifier(_BaseSparseAllSubsets, SparsePolyClassifierMixin):
    """Sparse all-subsets model for binary classification.
    Same surface as the reference class (sparse_all_subsets.py:394-519)."""
    _LOSSES = CLASSIFICATION_LOSSES

    def __init__(self, loss="squared_hinge", n_components=2, solver="pcd", beta=1, gamma=1, eta0=0.1,
                 mean=False, regularizer="omegati", tol=1e-6, warm_start=False, init_lambdas="ones",
                 max_iter=100, shuffle=False, verbose=False, callback=None, n_calls=10,
                 random_state=None):
        super().__init__(loss, n_components, solver, beta, gamma, eta0, mean, tol, regularizer,
                         warm_start, init_lambdas, max_iter, shuffle, verbose, callback, n_calls,
                         random_state)
