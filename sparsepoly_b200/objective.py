"""Objective of a fitted estimator, evaluated on the device.

The reference's update rules minimise

    sum_i loss(y_pred_i, y_i) + alpha/2 |w|^2 + beta/2 |P|^2 + gamma * Omega(P)

(alpha, beta, gamma times n_samples when mean=True; sparse_factorization_machines.py:181-188,
:265-272, sparse_all_subsets.py:86-91) but never evaluate it: the regularizers' `eval` methods
(regularizer/*.py) have no call site and, but for OmegaCS._eval, do not even compile under numba.
Parity "objective within 1e-9" therefore needs its own evaluator; this one runs the prediction
DP kernel and three deterministic device reductions (csrc/objective.cu) and returns the parts.
"""
import numpy as np
import torch

from . import _lib, solvers
from .dataset import DeviceDataset, _device, check_X, host_y

_f64 = torch.float64


def _targets(est, y):
    y = np.asarray(host_y(y))
    if hasattr(est, "label_binarizer_"):
        return est.label_binarizer_.transform(y).ravel().astype(np.float64)
    return np.ascontiguousarray(y, dtype=np.float64).ravel()


def objective(est, X, y):
    """Parts and total of the training objective of a fitted Sparse{FactorizationMachine,AllSubsets}
    {Regressor,Classifier} on (X, y): dict(loss, l2_w, l2_P, omega, total).  Order o of an FM's P_
    enters with degree `degree - o` (explicit lower orders, sparse_factorization_machines.py:207-225)."""
    from sklearn.exceptions import NotFittedError
    if not hasattr(est, "P_"):
        raise NotFittedError("Estimator not fitted.")
    dev = _device()
    _lib.check(_lib.load().sp_set_device(dev.index if dev.index is not None else 0))
    X = check_X(X, accept_sparse=["csr", "csc"], dtype=np.double)
    is_fm = hasattr(est, "degree")
    if is_fm:
        X = est._augment(X)
    n = X.shape[0]
    y_dev = torch.from_numpy(_targets(est, y)).to(dev)
    ds = DeviceDataset(X, need_csr=True, need_csc=False, device=dev)
    lams = torch.from_numpy(np.ascontiguousarray(est.lams_, dtype=np.float64)).to(dev)
    y_pred = torch.zeros(n, dtype=_f64, device=dev)
    scale = n if est.mean else 1
    if is_fm:
        P = torch.from_numpy(np.ascontiguousarray(est.P_)).to(dev)          # [n_orders, k, d]
        w = torch.from_numpy(np.ascontiguousarray(est.w_)).to(dev)
        est._device_output(ds, P, w, lams, y_pred, 1)
        orders = [(solvers.transpose(P[o]), est.degree - o) for o in range(P.shape[0])]
        alpha, beta, gamma = est.alpha * scale, est.beta * scale, est.gamma * scale
        l2_w = solvers.sqnorm(w) if est.fit_linear else torch.zeros(1, dtype=_f64, device=dev)
    else:
        P_dk = solvers.transpose(torch.from_numpy(np.ascontiguousarray(est.P_)).to(dev))
        solvers.poly_predict(ds, P_dk, lams, -1, out=y_pred)
        orders = [(P_dk, -1)]
        alpha, beta, gamma = 0.0, est.beta * scale, est.gamma * scale
        l2_w = torch.zeros(1, dtype=_f64, device=dev)
    loss = solvers.loss_sum(y_pred, y_dev, est.loss, n)
    l2_P = torch.zeros(1, dtype=_f64, device=dev)
    omega = torch.zeros(1, dtype=_f64, device=dev)
    for P_dk, deg in orders:
        l2_P += solvers.sqnorm(P_dk)
        omega += solvers.reg_eval(P_dk, est.regularizer, deg)
    parts = torch.cat([loss, l2_w, l2_P, omega]).cpu().numpy()             # one D2H of 4 doubles
    out = dict(loss=float(parts[0]), l2_w=float(parts[1]), l2_P=float(parts[2]), omega=float(parts[3]))
    out["total"] = out["loss"] + 0.5 * alpha * out["l2_w"] + 0.5 * beta * out["l2_P"] + gamma * out["omega"]
    return out
