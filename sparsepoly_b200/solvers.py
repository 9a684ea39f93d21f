"""Host-side drivers that launch the CUDA epochs (Python mirror of the reference's operator
boundary, SURVEY.md 8b).  Function names follow reference optimizer/*.py; every function works
on torch CUDA tensors that are mutated in place, exactly as the numba functions mutate numpy
arrays.  PyTorch is only the allocator / stream / collective provider here.
"""
import ctypes as C

import numpy as np
import torch

from . import _lib
from .dataset import SweepPlan, _ptr, _stream  # noqa: F401

_f64 = torch.float64


def _L():
    return _lib.load()


def rec_stride(degree):
    return int(_L().sp_rec_stride(int(degree)))


def transpose(t):
    """Device transpose of a 2-D fp64 tensor (sp_transpose_f64)."""
    rows, cols = t.shape
    out = torch.empty((cols, rows), dtype=_f64, device=t.device)
    _lib.check(_L().sp_transpose_f64(_ptr(t), _ptr(out), rows, cols, _stream()))
    return out


def transpose_batch(t):
    """Device transpose of every matrix of a 3-D fp64 tensor [batch, rows, cols] in one launch (sp_transpose_f64_batch)."""
    batch, rows, cols = t.shape
    out = torch.empty((batch, cols, rows), dtype=_f64, device=t.device)
    _lib.check(_L().sp_transpose_f64_batch(_ptr(t), _ptr(out), batch, rows, cols, _stream()))
    return out


def poly_predict(ds, P_dk, lams, degree, w=None, out=None, out_stride=1, accumulate=False):
    """kernels.poly_predict on device (kernels.py:140-153): out[i*stride] (+)= <w,x_i> +
    sum_s lams[s] K(P[:,s], x_i); degree=-1 selects the all-subsets kernel."""
    if out is None:
        out = torch.zeros(ds.n_samples * out_stride, dtype=_f64, device=ds.device)
    _lib.check(_L().sp_predict(ds.ref(), _ptr(P_dk), int(P_dk.shape[1]), _ptr(lams), int(degree),
                               _ptr(w), _ptr(out), int(out_stride), int(bool(accumulate)), _stream()))
    return out


def predict_multi(ds, models, k, degree, out_stride=1, accumulate=False):
    """poly_predict of every model of a ctypes SpPredictModel array (<= _lib.PREDICT_MAX_MODELS) in one launch."""
    _lib.check(_L().sp_predict_multi(ds.ref(), models, len(models), int(k), int(degree), int(out_stride),
                                     int(bool(accumulate)), _stream()))


def cd_linear_epoch(ds, plan, w, col_norm_sq, alpha, loss, rec, stride, viol):
    """cd_linear._cd_linear_epoch (cd_linear.py:8-33)."""
    _lib.check(_L().sp_cd_linear_epoch(ds.ref(), plan.ref(), _ptr(w), _ptr(col_norm_sq), float(alpha),
                                       _lib.LOSS_IDS[loss], _ptr(rec), int(stride), _ptr(viol),
                                       _stream()))


def pcd_epoch(ds, plan, P_kd, lams, degree, beta, gamma, eta, reg, loss, rec, stride, regstate, viol,
              indices_component):
    """pcd.pcd_epoch (pcd.py:71-137) / pcd_all.pcd_epoch (pcd_all.py:44-102, degree=-1)."""
    idx = np.ascontiguousarray(indices_component, dtype=np.int32)
    _lib.check(_L().sp_pcd_epoch(ds.ref(), plan.ref(), _ptr(P_kd), int(P_kd.shape[0]), _ptr(lams),
                                 int(degree), float(beta), float(gamma), float(eta),
                                 _lib.REG_IDS[reg], _lib.LOSS_IDS[loss], _ptr(rec), int(stride),
                                 _ptr(regstate), _ptr(viol),
                                 idx.ctypes.data_as(C.POINTER(C.c_int32)), _stream()))


def cd_linear_epoch_multi(ds, n_cta, threads, col_norm_sq, models, loss, stride):
    """cd_linear_epoch of every model of a ctypes SpPcdModel array in one launch (fit_many)."""
    _lib.check(_L().sp_cd_linear_epoch_multi(ds.ref(), int(n_cta), int(threads), _ptr(col_norm_sq), models,
                                             len(models), _lib.LOSS_IDS[loss], int(stride), _stream()))


def pcd_epoch_multi(ds, n_cta, threads, models, k, degree, loss, stride):
    """pcd_epoch of one order of every model of a ctypes SpPcdModel array; each launch covers all models
    (fit_many)."""
    _lib.check(_L().sp_pcd_epoch_multi(ds.ref(), int(n_cta), int(threads), models, len(models), int(k),
                                       int(degree), _lib.LOSS_IDS[loss], int(stride), _stream()))


def pbcd_epoch(ds, plan, P_dk, lams, degree, beta, gamma, eta, reg, loss, yrec, A, reg_norms, regstate,
               viol):
    """pbcd.pbcd_epoch (pbcd.py:82-148) / pbcd_all.pbcd_epoch (pbcd_all.py:68-132, degree=-1)."""
    _lib.check(_L().sp_pbcd_epoch(ds.ref(), plan.ref(), _ptr(P_dk), int(P_dk.shape[1]), _ptr(lams),
                                  int(degree), float(beta), float(gamma), float(eta),
                                  _lib.REG_IDS[reg], _lib.LOSS_IDS[loss], _ptr(yrec), _ptr(A),
                                  _ptr(reg_norms), _ptr(regstate), _ptr(viol), _stream()))


def pbcd_epoch_multi(ds, n_cta, threads, models, k, degree, loss):
    """pbcd_epoch of one order of every model of a ctypes SpPbcdModel array; each launch covers all models
    (fit_many)."""
    _lib.check(_L().sp_pbcd_epoch_multi(ds.ref(), int(n_cta), int(threads), models, len(models), int(k),
                                        int(degree), _lib.LOSS_IDS[loss], _stream()))


def get_eta(learning_rate, eta0, alpha, beta, power_t, it):
    """psgd._get_eta (psgd.py:9-22)."""
    a, b = C.c_double(), C.c_double()
    _lib.check(_L().sp_get_eta(int(learning_rate), float(eta0), float(alpha), float(beta),
                               float(power_t), int(it), C.byref(a), C.byref(b)))
    return a.value, b.value


def prox_work(d, k, device):
    return torch.empty(int(_L().sp_prox_work_doubles(int(d), int(k))), dtype=_f64, device=device)


def prox(P_dk, reg, strength, work):
    """regularizer.prox on one order (l1.py:50, l21.py:43, squaredl12.py:66, squaredl21.py:63)."""
    d, k = P_dk.shape
    _lib.check(_L().sp_prox(_ptr(P_dk), int(d), int(k), _lib.REG_IDS[reg], float(strength), _ptr(work),
                            _stream()))


def psgd_grad(ds, y, P_odk, w, lams, degree, loss, fit_linear, idx_samples, b0, b1, grad_P, grad_w, loss_sum):
    """psgd._pred + _update_grads for samples idx_samples[b0:b1] (psgd.py:47-91), dense-gradient path."""
    n_orders, _, k = P_odk.shape
    _lib.check(_L().sp_psgd_grad(ds.ref(), _ptr(y), _ptr(P_odk), int(n_orders), int(k), _ptr(w),
                                 _ptr(lams), int(degree), _lib.LOSS_IDS[loss], int(bool(fit_linear)),
                                 _ptr(idx_samples), int(b0), int(b1), _ptr(grad_P), _ptr(grad_w),
                                 _ptr(loss_sum), _stream()))


def psgd_step(P_odk, grad_P, w, grad_w, eta_P, eta_w, alpha, beta, batch, fit_linear):
    """SGD part of psgd._update_params + gradient zeroing (psgd.py:94-117, :195-196)."""
    n_orders, d, k = P_odk.shape
    _lib.check(_L().sp_psgd_step(_ptr(P_odk), _ptr(grad_P), _ptr(w), _ptr(grad_w), int(n_orders), int(d),
                                 int(k), float(eta_P), float(eta_w), float(alpha), float(beta),
                                 int(batch), int(bool(fit_linear)), _stream()))


PLANNED_REGS = ("l1", "squaredl12")     # prox = column-wise soft threshold: planned path (psgd_plan.cu)


def psgd_epoch(ds, y, P_odk, w, lams, degree, alpha, beta, gamma, reg, loss, grad_P, grad_w,
               idx_samples, fit_linear, eta0, learning_rate, power_t, batch_size, it, loss_sum, work,
               group=None):
    """psgd.psgd_epoch (psgd.py:125-199) on the dense-gradient path (any regularizer).  Returns the
    advanced `it`; the epoch's loss sum is accumulated into the device scalar loss_sum.

    With `group` (a torch.distributed process group of G ranks, each holding an equal shard of the
    samples) every rank contributes batch_size//G samples to each minibatch and the dense gradients are
    summed with one all-reduce before the (replicated) update.  l1 / squaredl12 fits do not come here:
    they run the planned path (psgd_planned_*), which shards over peer memory instead."""
    n_orders, d, k = P_odk.shape
    if group is None:
        it_c = C.c_int64(int(it))
        _lib.check(_L().sp_psgd_epoch(ds.ref(), _ptr(y), _ptr(P_odk), int(n_orders), int(k), _ptr(w),
                                      _ptr(lams), int(degree), float(alpha), float(beta), float(gamma),
                                      _lib.REG_IDS[reg], _lib.LOSS_IDS[loss], _ptr(grad_P),
                                      _ptr(grad_w), _ptr(idx_samples), int(bool(fit_linear)),
                                      float(eta0), int(learning_rate), float(power_t),
                                      int(batch_size), C.byref(it_c), _ptr(loss_sum), _ptr(work),
                                      _stream()))
        return it_c.value
    import torch.distributed as dist
    from .distributed import local_batches
    world = dist.get_world_size(group)
    for b0, b1, b_global in local_batches(ds.n_samples, batch_size, world):
        psgd_grad(ds, y, P_odk, w, lams, degree, loss, fit_linear, idx_samples, b0, b1, grad_P, grad_w, loss_sum)
        if fit_linear:
            dist.all_reduce(grad_w, group=group)
        dist.all_reduce(grad_P, group=group)
        eta_P, eta_w = get_eta(learning_rate, eta0, alpha, beta, power_t, it)
        strength = gamma * eta_P / (1 + eta_P * beta)
        psgd_step(P_odk, grad_P, w, grad_w, eta_P, eta_w, alpha, beta, b_global, fit_linear)
        for o in range(n_orders):
            prox(P_odk[o], reg, strength, work)
        it += 1
    return it


def psgd_planned_begin(ctx):
    """Start of a planned fit: the context's P / w hold the model, thresholds and scales are reset."""
    _lib.check(_L().sp_psgd_plan_begin(ctx.ref(), _stream()))


def psgd_planned_run(ctx, ds, plan, y, idx_samples, alpha, beta, gamma, eta0, learning_rate, power_t, it,
                     m_begin=0, m_end=None):
    """Minibatches [m_begin, m_end) of psgd.psgd_epoch (psgd.py:150-198) on the planned path; returns the
    advanced `it`."""
    it_c = C.c_int64(int(it))
    m_end = plan.n_minibatches if m_end is None else m_end
    _lib.check(_L().sp_psgd_plan_run(ctx.ref(), ds.ref(), plan.ref(), _ptr(y), _ptr(idx_samples), float(alpha),
                                     float(beta), float(gamma), float(eta0), int(learning_rate), float(power_t),
                                     int(m_begin), int(m_end), C.byref(it_c), _stream()))
    return it_c.value


def psgd_planned_solver_stats(ctx):
    """(prox calls, solved from the band, needed generic passes, band half-width) of the squared-l1,2 selection."""
    out = (C.c_double * 6)()
    _lib.check(_L().sp_psgd_plan_solver_stats(ctx.ref(), out, _stream()))
    return {"prox_calls": int(out[0]), "band_solves": int(out[1]), "generic_solves": int(out[2]), "band_half_width": out[3],
            "band_values_per_column_mean": out[4], "band_values_per_column_max": out[5]}


def psgd_planned_end(ctx, n_local, loss_sum, materialize):
    """End of an epoch: loss_sum[0] += the epoch's loss sum (fixed order); materialize=True turns the lazily
    scaled / thresholded storage back into the model."""
    _lib.check(_L().sp_psgd_plan_end(ctx.ref(), int(n_local), _ptr(loss_sum), int(bool(materialize)), _stream()))


def psgd_planned_read(ctx, P_okd, w):
    """The model the lazy frame represents into P_okd [n_orders, k, d] / w [d] (device); ctx is left as it was."""
    _lib.check(_L().sp_psgd_plan_read(ctx.ref(), _ptr(P_okd), _ptr(w), _stream()))


# ------------------------------------------------------------------------------ objective
def _sum_work(device):
    return torch.empty(int(_L().sp_sum_work_doubles()), dtype=_f64, device=device)


def loss_sum(y_pred, y, loss, n, pred_stride=1, y_stride=1):
    """sum_i loss(y_pred[i*pred_stride], y[i*y_stride]) (loss.py:19-20, :34-41, :61-65) as a
    1-element device tensor; the strides let it read the sweep records {y_pred, y, ...} in place."""
    out = torch.empty(1, dtype=_f64, device=y_pred.device)
    _lib.check(_L().sp_loss_sum(_ptr(y_pred), int(pred_stride), _ptr(y), int(y_stride), int(n),
                                _lib.LOSS_IDS[loss], _ptr(_sum_work(y_pred.device)), _ptr(out), _stream()))
    return out


def sqnorm(t):
    """sum of squares of a contiguous fp64 device tensor (1-element device tensor)."""
    out = torch.empty(1, dtype=_f64, device=t.device)
    _lib.check(_L().sp_sqnorm(_ptr(t), int(t.numel()), _ptr(_sum_work(t.device)), _ptr(out), _stream()))
    return out


def reg_eval(P_dk, reg, degree):
    """Omega(P) of one order, P_dk feature-major [d,k] (the regularizer classes' `eval`:
    l1.py:17-18, l21.py:19-21, squaredl12.py:20-22, squaredl21.py:23-25, omegati.py:19-47,
    omegacs.py:22-39); degree=-1: all-subsets.  1-element device tensor."""
    d, k = P_dk.shape
    out = torch.empty(1, dtype=_f64, device=P_dk.device)
    work = torch.empty(int(_L().sp_reg_eval_work_doubles(int(d), int(k))), dtype=_f64, device=P_dk.device)
    _lib.check(_L().sp_reg_eval(_ptr(P_dk), int(d), int(k), _lib.REG_IDS[reg], int(degree), _ptr(work),
                                _ptr(out), _stream()))
    return out


def loss_sum_multi(entries, n, work, pred_stride=1, y_stride=1):
    """loss_sum of every entry of a ctypes SpLossEntry array (<= _lib.OBJECTIVE_MAX_ENTRIES); work holds
    len(entries) * sp_sum_work_doubles() doubles."""
    _lib.check(_L().sp_loss_sum_multi(entries, len(entries), int(pred_stride), int(y_stride), int(n), _ptr(work),
                                      _stream()))


def sqnorm_multi(entries, length, work):
    """sqnorm of every entry of a ctypes SpSqnormEntry array, all of `length` doubles."""
    _lib.check(_L().sp_sqnorm_multi(entries, len(entries), int(length), _ptr(work), _stream()))


def reg_eval_multi(entries, d, k, degree, work):
    """reg_eval of every entry of a ctypes SpRegEntry array, all [d,k] at this degree; work holds
    len(entries) * sp_reg_eval_work_doubles(d, k) doubles."""
    _lib.check(_L().sp_reg_eval_multi(entries, len(entries), int(d), int(k), int(degree), _ptr(work), _stream()))


def sum_work_doubles():
    return int(_L().sp_sum_work_doubles())


def reg_eval_work_doubles(d, k):
    return int(_L().sp_reg_eval_work_doubles(int(d), int(k)))
