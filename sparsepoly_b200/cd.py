"""The coordinate-descent driver of the pcd / pbcd fits: a single fit (factorization machine or all-subsets) and a
fit_many call run their epochs through this module.

  * CdModel: one model's device state -- records, P in the layout its solver trains, scratch, coordinate orders;
  * sub_epochs: the sub-epochs of one epoch, in the reference's order (sparse_factorization_machines.py:196-243,
    sparse_all_subsets.py:104-133 / :160-199);
  * run_epoch: one epoch of a list of models, through one launch function per sub-epoch kind;
  * stopping_loop: the stopping rule (violation sum < tol, callback, max_iter) over a list of models;
  * setup: the (epoch, sync) pair of a single fit, on its own sweep plans.
"""
import contextlib
import ctypes as C
import io
import warnings

import numpy as np
import torch

from . import _lib, solvers
from .dataset import DeviceDataset, SweepPlan

_f64 = torch.float64


def sub_epochs(est):
    """(kind, degree, order of P) of every sub-epoch of one epoch, in order: linear CD (kind "linear", on w), the
    explicit lower orders ascending (P[degree - deg]), the top order (P[0]).  kind is "linear" or est.solver."""
    if not hasattr(est, "degree"):
        return [(est.solver, -1, 0)]
    m = est.degree
    subs = [("linear", None, None)] if est.fit_linear else []
    if est.fit_lower == "explicit":
        subs += [(est.solver, deg, m - deg) for deg in range(2, m)]
    return subs + [(est.solver, m, 0)]


class CdModel:
    """Device state of one pcd or pbcd model: the sample records {y_pred, y, ...} (stride doubles per sample) with the
    initial prediction, P [n_orders, k, d] (pcd) or feature-major [n_orders, d, k] (pbcd; all-subsets: one order),
    w, lams, the regularizer state, the violation sum (`viol`, one double of the caller's), pbcd's A cache and row
    norms, and the feature / component orders that shuffle() redraws from rng and sets on every plan of `plans`."""

    def __init__(self, est, ds, y, stride, plans, viol, rng):
        self.est, self.plans, self.viol, self.rng = est, plans, viol, rng
        self.fm, self.pbcd = hasattr(est, "degree"), est.solver == "pbcd"
        dev, n, d, k = ds.device, ds.n_samples, ds.n_features, est.n_components
        self.rec = torch.zeros(n * stride, dtype=_f64, device=dev)
        self.rec[1::stride] = torch.from_numpy(y).to(dev)
        P = torch.from_numpy(np.ascontiguousarray(est.P_)).to(dev)
        self.lams = torch.from_numpy(np.ascontiguousarray(est.lams_, dtype=np.float64)).to(dev)
        if self.fm:
            self.w = torch.from_numpy(np.ascontiguousarray(est.w_)).to(dev)
            est._device_output(ds, P, self.w, self.lams, self.rec, stride)          # y_pred -> rec[0::stride]
            self.alpha, self.beta, self.gamma = est._scaled(n)
            self.P = solvers.transpose_batch(P) if self.pbcd else P
        else:
            self.w = None
            P_dk = solvers.transpose_batch(P.view(1, k, d))
            solvers.poly_predict(ds, P_dk[0], self.lams, -1, out=self.rec, out_stride=stride)
            self.alpha = 0.0
            self.beta, self.gamma = (n * est.beta, n * est.gamma) if est.mean else (est.beta, est.gamma)
            self.P = P_dk if self.pbcd else P.view(1, k, d)
        self.regstate = torch.zeros(16, dtype=_f64, device=dev)
        self.idx_feat = np.arange(d, dtype=np.int32)
        self.idx_comp = None if self.pbcd else np.arange(k, dtype=np.int32)
        if self.pbcd:
            self.A = torch.empty(max(n * (est.degree - 1 if self.fm else 1) * k, 1), dtype=_f64, device=dev)
            self.reg_norms = torch.zeros(max(d, 1), dtype=_f64, device=dev)
        for plan in plans:
            plan.set_order(self.idx_feat)

    def shuffle(self):
        """The draws of one epoch: pcd shuffles the components then the features, pbcd the features only."""
        if self.idx_comp is not None:
            self.rng.shuffle(self.idx_comp)
        self.rng.shuffle(self.idx_feat)
        for plan in self.plans:
            plan.set_order(self.idx_feat)

    def sync(self):
        """The device model into the estimator's P_ / w_, in place."""
        P = solvers.transpose_batch(self.P) if self.pbcd else self.P
        self.est.P_[...] = P.cpu().numpy().reshape(self.est.P_.shape)
        if self.w is not None:
            self.est.w_[...] = self.w.cpu().numpy()

    def entry(self, kind, order):
        """The sp_pcd_model ("linear", "pcd") or sp_pbcd_model ("pbcd") table entry of this model's sub-epoch on
        P[order] (w for "linear"), on its first plan."""
        s, e = self.plans[0].struct, self.est
        if kind == "pbcd":
            return _lib.SpPbcdModel(pos_ptr=s.pos_ptr, flag_idx=s.flag_idx, idx_feat=s.idx_feat,
                                    P=self.P[order].data_ptr(), lams=self.lams.data_ptr(), beta=float(self.beta),
                                    gamma=float(self.gamma), eta=float(e.eta0), reg=_lib.REG_IDS[e.regularizer],
                                    yrec=self.rec.data_ptr(), A=self.A.data_ptr(), reg_norms=self.reg_norms.data_ptr(),
                                    regstate=self.regstate.data_ptr(), viol=self.viol.data_ptr())
        linear = kind == "linear"
        idx_comp = None if self.idx_comp is None else self.idx_comp.ctypes.data_as(C.POINTER(C.c_int32))
        return _lib.SpPcdModel(pos_ptr=s.pos_ptr, flag_idx=s.flag_idx, idx_feat=s.idx_feat, pos_conf=s.pos_conf,
                               P=(self.w if linear else self.P[order]).data_ptr(), lams=self.lams.data_ptr(),
                               ab=float(self.alpha if linear else self.beta), gamma=float(self.gamma),
                               eta=float(e.eta0), reg=_lib.REG_IDS[e.regularizer], rec=self.rec.data_ptr(),
                               regstate=self.regstate.data_ptr(), viol=self.viol.data_ptr(), idx_comp_host=idx_comp)


def run_epoch(models, viol, launch):
    """One epoch of `models` (all of one estimator configuration): viol (holding every model's violation sum) is
    zeroed, the shuffling models draw their orders, then every sub-epoch runs as launch[kind](models, degree, order)."""
    viol.zero_()
    for m in models:
        if m.est.shuffle:
            m.shuffle()
    for kind, deg, order in sub_epochs(models[0].est):
        launch[kind](models, deg, order)


def stopping_loop(ests, syncs, epoch, buffered=False):
    """Run epochs until every model has stopped and return the models' converged flags.

    epoch(active) runs one epoch of the models whose indices are in `active` and returns their violation sums.  A
    model stops when its callback returns non-None (called every n_calls epochs after syncs[i]()), when its violation
    sum is below tol (converged) or after max_iter epochs.  At the end every model is synced, its n_iter_ is its last
    0-based epoch and an unconverged model warns.  buffered=True holds each model's verbose lines until then."""
    outs = [io.StringIO() if buffered else None for _ in ests]
    last, converged = [0] * len(ests), [False] * len(ests)
    active = [i for i, e in enumerate(ests) if e.max_iter > 0]
    it = 0
    while active:
        running = []
        for i, v in zip(active, epoch(active)):
            e = ests[i]
            last[i] = it
            with contextlib.redirect_stdout(outs[i]) if buffered else contextlib.nullcontext():
                stop = e._after_epoch(it, v, "Iteration {} violation sum {}", syncs[i])
                if not stop and v < e.tol:
                    if e.verbose:
                        print(f"Converged at iteration {it+1}")
                    converged[i] = stop = True
            if not stop and it + 1 < e.max_iter:
                running.append(i)
        active = running
        it += 1
    for i, e in enumerate(ests):
        syncs[i]()
        e.n_iter_ = last[i]
        if buffered:
            print(outs[i].getvalue(), end="")
        if not converged[i]:
            warnings.warn("Objective did not converge. Increase max_iter.")
    return converged


def setup(est, X, y, rng, dev):
    """Move a single pcd / pbcd fit to the device and return (epoch, sync): epoch(read_back=True) runs one epoch and
    returns the violation sum (None with read_back=False), sync() writes P_ / w_.  Sets est._h2d_bytes and
    est._dev_state (ds, plan of the top order, plan_lin of the linear sub-epoch, rec, stride, P, w).

    pcd runs every sub-epoch on one plan; pbcd runs each order on a plan of its own record shape and the linear
    sub-epoch on a pcd plan of stride 2."""
    k, pbcd = est.n_components, est.solver == "pbcd"
    ds = DeviceDataset(X, need_csr=True, need_csc=True, device=dev)
    est._h2d_bytes = ds.h2d_bytes + y.nbytes + est.P_.nbytes + (est.w_.nbytes if hasattr(est, "w_") else 0)
    subs = sub_epochs(est)
    stride = 2 if pbcd else solvers.rec_stride(subs[-1][1])             # (the top order's record shape)
    if pbcd:
        plans = {(kind, deg): (SweepPlan(ds, "pcd", rec_stride=2) if kind == "linear"
                               else SweepPlan(ds, "pbcd", pbcd_shape=(deg, k))) for kind, deg, _ in subs}
    else:
        plan = SweepPlan(ds, "pcd", rec_stride=stride)
        plans = {(kind, deg): plan for kind, deg, _ in subs}
    viol = torch.zeros(1, dtype=_f64, device=dev)
    m = CdModel(est, ds, y, stride, list(dict.fromkeys(plans.values())), viol, rng)
    col_norm_sq = ds.col_norm_sq() if subs[0][0] == "linear" else None
    est._dev_state = dict(ds=ds, plan=plans[subs[-1][:2]], plan_lin=plans.get(("linear", None)), rec=m.rec,
                          stride=stride, P=m.P if m.fm else m.P[0], w=m.w)
    launch = {
        "linear": lambda _, deg, o: solvers.cd_linear_epoch(ds, plans["linear", deg], m.w, col_norm_sq, m.alpha,
                                                            est.loss, m.rec, stride, viol),
        "pcd": lambda _, deg, o: solvers.pcd_epoch(ds, plans["pcd", deg], m.P[o], m.lams, deg, m.beta, m.gamma,
                                                   est.eta0, est.regularizer, est.loss, m.rec, stride, m.regstate,
                                                   viol, m.idx_comp),
        "pbcd": lambda _, deg, o: solvers.pbcd_epoch(ds, plans["pbcd", deg], m.P[o], m.lams, deg, m.beta, m.gamma,
                                                     est.eta0, est.regularizer, est.loss, m.rec, m.A, m.reg_norms,
                                                     m.regstate, viol),
    }

    def epoch(read_back=True):
        run_epoch([m], viol, launch)
        return viol.item() if read_back else None

    return epoch, m.sync
