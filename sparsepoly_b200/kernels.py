"""Device versions of reference sparsepoly/kernels.py (same function names and arguments).

The reference builds dense n x k Gram matrices with power-sum identities on the host
(kernels.py:91-114); here one CSR row kernel runs the degree-m ANOVA / all-subsets dynamic
program per (sample, component)."""
import numpy as np
import torch

from . import _lib
from .dataset import DeviceDataset, _device, _ptr, _stream, check_X, is_device_input


def _gram(X, P, degree):
    dev = _device()
    if is_device_input(X):              # (host X goes to DeviceDataset as it is, as before)
        X = check_X(X)
    ds = DeviceDataset(X, need_csr=True, need_csc=False, device=dev)
    P = np.ascontiguousarray(np.asarray(P, dtype=np.float64))
    P_dk = torch.from_numpy(np.ascontiguousarray(P.T)).to(dev)
    K = torch.empty((ds.n_samples, P.shape[0]), dtype=torch.float64, device=dev)
    _lib.check(_lib.load().sp_kernel_matrix(ds.ref(), _ptr(P_dk), int(P.shape[0]), int(degree), _ptr(K),
                                            _stream()))
    return K.cpu().numpy()


def anova_kernel(X, P, degree=2):
    """K_A(x, p) = sum_{j1<...<jm} prod_t x_jt p_jt  (kernels.py:71-115).  Returns [n, k]."""
    return _gram(X, P, degree)


def all_subsets_kernel(X, P):
    """K(x, p) = prod_j (1 + x_j p_j)  (kernels.py:118-137)."""
    return _gram(X, P, -1)


def homogeneous_kernel(X, P, degree=2):
    """K_P(x, p) = <x, p> ^ degree  (kernels.py:50-68): the degree-1 ANOVA kernel is the inner product."""
    return _gram(X, P, 1) ** degree


def poly_predict(X, P, lams, kernel, degree=2):
    """np.dot(K, lams)  (kernels.py:140-153); kernel in {'anova', 'poly', 'all-subsets'}."""
    if kernel == "anova":
        K = anova_kernel(X, P, degree)
    elif kernel == "poly":
        K = homogeneous_kernel(X, P, degree)
    elif kernel == "all-subsets":
        K = all_subsets_kernel(X, P)
    else:
        raise ValueError(("Unsuppported kernel: {}. Use one of "
                          "{{'anova'|'poly'|'all-subsets'}}").format(kernel))
    return np.dot(K, lams)
