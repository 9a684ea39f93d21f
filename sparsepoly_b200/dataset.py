"""Device-resident design matrix (replaces reference sparsepoly/dataset.py).

The reference wraps scipy CSR/CSC (or dense) arrays in numba jitclasses handing out row /
column slices (dataset.py:69-116).  Here the matrix lives in HBM in BOTH layouts as int32 /
fp64 torch tensors (PyTorch only holds the memory); kernels read coalesced row streams (CSR:
prediction, cache precompute, psgd) and column streams (CSC: coordinate sweeps).  Dense input
is stored with every entry, like the reference's ContiguousDataset / FortranDataset
(dataset.py:18-57).
"""
import ctypes as C
import os

import numpy as np
import scipy.sparse as sp
import torch
from sklearn.utils.validation import _check_y, check_array, check_consistent_length
from sklearn.utils.validation import check_X_y as _sk_check_X_y

from . import _lib


def _device(device=None):
    if not torch.cuda.is_available():
        raise RuntimeError("sparsepoly_b200 needs a CUDA device (there is no CPU fallback)")
    if device is None:
        device = torch.device("cuda", torch.cuda.current_device())
    return torch.device(device)


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def _h2d(a, device, pin=False):
    t = torch.from_numpy(np.ascontiguousarray(a))
    if pin:
        t = t.pin_memory()
    return t.to(device, non_blocking=pin)


def host_csr(X):
    """(indptr, indices, data) with sorted, duplicate-free rows; dense X keeps every entry."""
    if sp.issparse(X):
        Xr = sp.csr_matrix(X, dtype=np.float64, copy=False)
        if not Xr.has_canonical_format:
            Xr = Xr.copy()
            Xr.sum_duplicates()
        if Xr.nnz >= 2 ** 31:
            raise ValueError("nnz >= 2^31 is not supported (int32 indptr, reference dataset.py:60-66)")
        return (Xr.indptr.astype(np.int32, copy=False), Xr.indices.astype(np.int32, copy=False),
                Xr.data.astype(np.float64, copy=False))
    X = np.asarray(X, dtype=np.float64)
    n, d = X.shape
    if n * d >= 2 ** 31:
        raise ValueError("dense input with n_samples * n_features >= 2^31 is not supported (int32 indptr, reference "
                         "dataset.py:60-66); pass a scipy sparse matrix")
    indptr = (np.arange(n + 1, dtype=np.int64) * d).astype(np.int32)
    indices = np.tile(np.arange(d, dtype=np.int32), n)
    return indptr, indices, np.ascontiguousarray(X).reshape(-1)


def host_csc(X):
    if sp.issparse(X):
        Xc = sp.csc_matrix(X, dtype=np.float64, copy=False)
        if not Xc.has_canonical_format:
            Xc = Xc.copy()
            Xc.sum_duplicates()
        if Xc.nnz >= 2 ** 31:
            raise ValueError("nnz >= 2^31 is not supported (int32 indptr, reference dataset.py:60-66)")
        return (Xc.indptr.astype(np.int32, copy=False), Xc.indices.astype(np.int32, copy=False),
                Xc.data.astype(np.float64, copy=False))
    X = np.asarray(X, dtype=np.float64)
    n, d = X.shape
    if n * d >= 2 ** 31:
        raise ValueError("dense input with n_samples * n_features >= 2^31 is not supported (int32 indptr, reference "
                         "dataset.py:60-66); pass a scipy sparse matrix")
    indptr = (np.arange(d + 1, dtype=np.int64) * n).astype(np.int32)
    indices = np.tile(np.arange(n, dtype=np.int32), d)
    return indptr, indices, np.ascontiguousarray(X.T).reshape(-1)


_NO_ROW = 2 ** 63 - 1          # a "first row" entry of sp_csr_prepare's report that found nothing
_REPORT = dict(decreasing=0, indptr0=1, indptrn=2, range=3, nan=4, inf=5, n_unsorted=6, unsorted=7)


def is_device_input(X):
    """A CUDA tensor, or the DeviceCSR check_X made of one."""
    return isinstance(X, DeviceCSR) or (isinstance(X, torch.Tensor) and X.is_cuda)


def host_y(y):
    """Targets on the host: a torch tensor (on any device) becomes a numpy array; anything else is returned as is."""
    return y.detach().cpu().numpy() if isinstance(y, torch.Tensor) else y


class DeviceCSR:
    """A CUDA design matrix after check_X: the CSR host_csr gives for the same matrix (sorted, duplicate-free rows,
    int32 indptr / indices, fp64 data), on the device.  Canonical int32 / fp64 input is the caller's own tensors."""

    def __init__(self, shape, indptr, indices, data, dense):
        self.shape = (int(shape[0]), int(shape[1]))
        self.indptr, self.indices, self.data = indptr, indices, data
        self.nnz = int(data.numel())
        self.dense = dense              # from a strided tensor: every entry is stored

    def augment(self, n_dummy):
        """add_dummy_feature applied n_dummy times: columns 0..n_dummy-1 of ones, the others shifted by n_dummy."""
        if n_dummy == 0:
            return self
        n, d = self.shape
        _check_stored(self.nnz + n * n_dummy, self.dense)
        out = _alloc_csr(n, self.nnz + n * n_dummy, self.data.device)
        _run_prepare(n, d, self.indptr, self.indices, self.data, (0, 0), n_dummy, out)
        return DeviceCSR((n, d + n_dummy), *out, self.dense)


def _check_stored(stored, dense):
    if stored < 2 ** 31:
        return
    if dense:
        raise ValueError("dense input with n_samples * n_features >= 2^31 is not supported (int32 indptr, reference "
                         "dataset.py:60-66); pass a scipy sparse matrix")
    raise ValueError("nnz >= 2^31 is not supported (int32 indptr, reference dataset.py:60-66)")


def _alloc_csr(n, nnz, dev):
    return (torch.empty(n + 1, dtype=torch.int32, device=dev), torch.empty(nnz, dtype=torch.int32, device=dev),
            torch.empty(nnz, dtype=torch.float64, device=dev))


def _run_prepare(n, d, indptr, indices, values, strides, n_dummy, out=None):
    """sp_csr_prepare (indptr None: dense strided values); returns the report tensor (still on the device)."""
    report = torch.empty(_lib.CSR_REPORT_LEN, dtype=torch.int64, device=values.device)
    o = out if out is not None else (None, None, None)
    _lib.check(_lib.load().sp_csr_prepare(
        n, d, int(values.numel()), _ptr(indptr), int(indptr is not None and indptr.dtype == torch.int64),
        _ptr(indices), int(indices is not None and indices.dtype == torch.int64), _ptr(values),
        int(values.dtype == torch.float64), int(strides[0]), int(strides[1]), int(n_dummy), _ptr(o[0]), _ptr(o[1]),
        _ptr(o[2]), _ptr(report), _stream()))
    return report


def _raise_on_report(r, n_cols, dense, nnz, input_name):
    name = f" {input_name}" if input_name else ""
    if not dense:
        if r[_REPORT["decreasing"]] != _NO_ROW:
            raise ValueError(f"X: indptr decreases at row {r[_REPORT['decreasing']]} "
                             "(indptr[row + 1] < indptr[row])")
        if r[_REPORT["indptr0"]] != 0:
            raise ValueError(f"X: indptr[0] is {r[_REPORT['indptr0']]}, not 0")
        if r[_REPORT["indptrn"]] != nnz:
            raise ValueError(f"X: indptr[-1] is {r[_REPORT['indptrn']]} but X stores {nnz} entries")
        if r[_REPORT["range"]] != _NO_ROW:
            raise ValueError(f"X: a column index outside [0, {n_cols}) in row {r[_REPORT['range']]}")
    # sklearn's wording (_assert_all_finite): NaN wins over infinity
    if r[_REPORT["nan"]] != _NO_ROW:
        raise ValueError(f"Input{name} contains NaN. First in row {r[_REPORT['nan']]}.")
    if r[_REPORT["inf"]] != _NO_ROW:
        raise ValueError(f"Input{name} contains infinity or a value too large for dtype('float64'). "
                         f"First in row {r[_REPORT['inf']]}.")


def _canonical(n, d, indptr, indices, data):
    """Sorted, duplicate-free rows of a CSR: stable sort of the (row, column) keys, then every run of equal keys summed
    left to right (sp_csr_sum_runs), as scipy's sum_duplicates; sums that come to zero stay stored."""
    nnz, dev = int(data.numel()), data.device
    counts = (indptr[1:] - indptr[:-1]).to(torch.int64)
    rows = torch.repeat_interleave(torch.arange(n, dtype=torch.int64, device=dev), counts, output_size=nnz)
    keys, perm = torch.sort(rows * d + indices.to(torch.int64), stable=True)
    del rows
    head = torch.ones(nnz, dtype=torch.bool, device=dev)
    head[1:] = keys[1:] != keys[:-1]
    runs_before = torch.zeros(nnz + 1, dtype=torch.int64, device=dev)       # runs_before[p]: heads in [0, p)
    torch.cumsum(head, 0, out=runs_before[1:])
    del head
    n_runs = int(runs_before[-1].item())
    out_indices = torch.empty(n_runs, dtype=torch.int32, device=dev)
    out_data = torch.empty(n_runs, dtype=torch.float64, device=dev)
    _lib.check(_lib.load().sp_csr_sum_runs(nnz, _ptr(keys), _ptr(perm), _ptr(data), _ptr(runs_before), d,
                                           _ptr(out_indices), _ptr(out_data), _stream()))
    return runs_before[indptr.to(torch.int64)].to(torch.int32), out_indices, out_data


def device_csr(X, ensure_min_samples=1, ensure_min_features=1, input_name=""):
    """Check a CUDA X (torch.sparse_csr or strided, 2-D, float32 / float64 values, int32 / int64 indices) on the
    device and return it as a DeviceCSR: one sp_csr_prepare pass, one small report read back; rows with unsorted or
    repeated columns are canonicalised on the device.  A DeviceCSR is already checked and is returned as it is."""
    if isinstance(X, DeviceCSR):
        return X
    dev = torch.device("cuda", torch.cuda.current_device())
    if X.device != dev:
        raise ValueError(f"X is on {X.device} but the current CUDA device is {dev}; move X there or make its device "
                         "current (torch.cuda.set_device)")
    floats = (torch.float32, torch.float64)
    if X.layout == torch.sparse_csr:
        if X.dim() != 2 or X.dense_dim() != 0:
            raise ValueError(f"a CUDA sparse CSR X must be 2-D, not batched and without dense dimensions; got shape "
                             f"{tuple(X.shape)} with {X.dense_dim()} dense dimension(s)")
        indptr, indices, values = X.crow_indices(), X.col_indices(), X.values()
        if indptr.dtype not in (torch.int32, torch.int64) or indices.dtype not in (torch.int32, torch.int64):
            raise ValueError(f"a CUDA sparse CSR X needs int32 or int64 indices, got {indices.dtype}")
        if values.dtype not in floats:
            raise ValueError(f"a CUDA X needs float32 or float64 values, got {values.dtype}")
        indptr, indices, values = indptr.contiguous(), indices.contiguous(), values.contiguous()
        if indices.numel() != values.numel() or indptr.numel() != X.shape[0] + 1:
            raise ValueError(f"X: {indptr.numel()} indptr entries, {indices.numel()} indices and {values.numel()} "
                             f"values do not form a CSR matrix of shape {tuple(X.shape)}")
        dense, strides = False, (0, 0)
    elif X.layout == torch.strided:
        if X.dim() != 2:
            raise ValueError(f"a CUDA X must be 2-D; got shape {tuple(X.shape)}")
        if X.dtype not in floats:
            raise ValueError(f"a CUDA X needs float32 or float64 values, got {X.dtype}")
        indptr = indices = None
        values, dense, strides = X, True, X.stride()
    else:
        raise ValueError(f"a CUDA X must be a torch.sparse_csr or a strided (dense) tensor, got layout {X.layout}; "
                         "convert it with .to_sparse_csr()")
    n, d = int(X.shape[0]), int(X.shape[1])
    if n < ensure_min_samples:
        raise ValueError(f"Found array with {n} sample(s) (shape={(n, d)}) while a minimum of {ensure_min_samples} "
                         "is required.")
    if d < ensure_min_features:
        raise ValueError(f"Found array with {d} feature(s) (shape={(n, d)}) while a minimum of {ensure_min_features} "
                         "is required.")
    nnz = n * d if dense else int(values.numel())
    _check_stored(nnz, dense)
    wrap = not dense and indptr.dtype == indices.dtype == torch.int32 and values.dtype == torch.float64
    out = None if wrap else _alloc_csr(n, nnz, dev)
    r = _run_prepare(n, d, indptr, indices, values, strides, 0, out).tolist()      # the one D2H of the check
    _raise_on_report(r, d, dense, nnz, input_name)
    if r[_REPORT["n_unsorted"]]:
        if out is None:
            out = _alloc_csr(n, nnz, dev)
            _run_prepare(n, d, indptr, indices, values, strides, 0, out)
        out = _canonical(n, d, *out)
    return DeviceCSR((n, d), *(out if out is not None else (indptr, indices, values)), dense)


def check_X(X, **check_array_kwargs):
    """The one place that decides between the host and the device path: a CUDA tensor is checked and converted on the
    device (device_csr; ensure_min_samples / ensure_min_features / input_name are honoured, the result is always
    fp64), anything else goes through sklearn's check_array with the same arguments."""
    if not is_device_input(X):
        return check_array(X, **check_array_kwargs)
    keys = ("ensure_min_samples", "ensure_min_features", "input_name")
    return device_csr(X, **{k: v for k, v in check_array_kwargs.items() if k in keys})


def check_X_y(X, y, **check_X_y_kwargs):
    """sklearn's check_X_y for host X; for a CUDA X, check_X then sklearn's checks of y (y_numeric as given)."""
    y = host_y(y)
    if not is_device_input(X):
        return _sk_check_X_y(X, y, **check_X_y_kwargs)
    X = device_csr(X, input_name="X")
    y = _check_y(y, multi_output=check_X_y_kwargs.get("multi_output", False),
                 y_numeric=check_X_y_kwargs.get("y_numeric", False))
    check_consistent_length(X, y)
    return X, y


def csr_to_csc_device(n, d, indptr, indices, data):
    """CSC (indptr, indices, data) of a canonical device CSR matrix: stable sort of the nonzeros by
    column keeps the rows ascending inside every column, i.e. scipy's canonical CSC, bit for bit."""
    nnz = int(data.numel())
    dev = data.device
    if nnz == 0:
        return (torch.zeros(d + 1, dtype=torch.int32, device=dev), torch.zeros(0, dtype=torch.int32, device=dev),
                torch.zeros(0, dtype=torch.float64, device=dev))
    counts = (indptr[1:] - indptr[:-1]).to(torch.int64)
    rows = torch.repeat_interleave(torch.arange(n, dtype=torch.int32, device=dev), counts, output_size=nnz)
    _, perm = torch.sort(indices, stable=True)
    csc_indices = rows[perm]
    csc_data = data[perm]
    del rows
    colcount = torch.bincount(indices, minlength=d)
    csc_indptr = torch.zeros(d + 1, dtype=torch.int32, device=dev)
    csc_indptr[1:] = torch.cumsum(colcount, 0).to(torch.int32)
    return csc_indptr, csc_indices.contiguous(), csc_data.contiguous()


class DeviceDataset:
    """CSR and/or CSC copy of X in device memory + the sp_dataset struct handed to the C ABI."""

    def __init__(self, X, need_csr=True, need_csc=True, device=None, pin=False, hot_features=True):
        self.device = _device(device)
        self.n_samples, self.n_features = int(X.shape[0]), int(X.shape[1])
        self.h2d_bytes = 0
        self.csr = self.csc = None
        if isinstance(X, DeviceCSR):          # (check_X of a CUDA X: already on the device, nothing to copy)
            csr = (X.indptr, X.indices, X.data)
            if need_csc:
                self.csc = csr_to_csc_device(self.n_samples, self.n_features, *csr)
            self.csr = csr if need_csr else None
        elif need_csr:
            self.csr = tuple(_h2d(a, self.device, pin) for a in host_csr(X))
            self.h2d_bytes += sum(t.numel() * t.element_size() for t in self.csr)
        if need_csc and self.csc is None:
            if need_csr and sp.issparse(X):
                # transpose on the device (the reference's get_dataset does a host tocsc(),
                # dataset.py:119-134; at C2 that is ~1 s of scipy against a few ms here)
                self.csc = csr_to_csc_device(self.n_samples, self.n_features, *self.csr)
            else:
                self.csc = tuple(_h2d(a, self.device, pin) for a in host_csc(X))
                self.h2d_bytes += sum(t.numel() * t.element_size() for t in self.csc)
        ref = self.csr if self.csr is not None else self.csc
        self.nnz = int(ref[2].numel())
        s = _lib.SpDataset()
        s.n_samples, s.n_features, s.nnz = self.n_samples, self.n_features, self.nnz
        if self.csr is not None:
            s.csr_indptr, s.csr_indices, s.csr_data = (t.data_ptr() for t in self.csr)
        if self.csc is not None:
            s.csc_indptr, s.csc_indices, s.csc_data = (t.data_ptr() for t in self.csc)
        self.struct = s
        if self.csr is not None and not need_csc and hot_features:
            self.mark_hot_features()

    def max_row_nnz(self):
        ip = self.csr[0]
        return int((ip[1:] - ip[:-1]).max().item()) if self.n_samples else 0

    def mark_hot_features(self, min_density=1.0 / 16, max_hot=16):
        """Dense features (present in >= 1/16 of the rows): sp_psgd_grad pre-reduces their gradient
        rows per warp (they would otherwise take one same-address atomic per sample)."""
        if self.csr is None or self.nnz == 0:
            return
        cnt = torch.bincount(self.csr[1], minlength=self.n_features)
        top = torch.topk(cnt, min(max_hot, self.n_features))
        keep = top.values.to(torch.float64) >= min_density * self.n_samples
        feats = top.indices[keep].to(torch.int32)
        if feats.numel() == 0:
            return
        self.hot_feat = feats.contiguous()
        self.feat_hot = torch.full((self.n_features,), -1, dtype=torch.int8, device=self.device)
        self.feat_hot[feats.long()] = torch.arange(feats.numel(), dtype=torch.int8, device=self.device)
        self.struct.feat_hot = self.feat_hot.data_ptr()
        self.struct.hot_feat = self.hot_feat.data_ptr()
        self.struct.n_hot_feat = int(feats.numel())

    def adopt_hot_features(self, other):
        """Reuse another dataset's dense-feature table (same feature space)."""
        if getattr(other, "feat_hot", None) is not None:
            self.feat_hot, self.hot_feat = other.feat_hot, other.hot_feat
            self.struct.feat_hot = other.struct.feat_hot
            self.struct.hot_feat = other.struct.hot_feat
            self.struct.n_hot_feat = other.struct.n_hot_feat

    @classmethod
    def from_device_csr(cls, n_samples, n_features, indptr, indices, data):
        """Wrap CSR tensors that already live on the device (no copy)."""
        self = cls.__new__(cls)
        self.device = data.device
        self.n_samples, self.n_features = int(n_samples), int(n_features)
        self.csr, self.csc = (indptr, indices, data), None
        self.nnz = int(data.numel())
        self.h2d_bytes = 0
        s = _lib.SpDataset()
        s.n_samples, s.n_features, s.nnz = self.n_samples, self.n_features, self.nnz
        s.csr_indptr, s.csr_indices, s.csr_data = indptr.data_ptr(), indices.data_ptr(), data.data_ptr()
        self.struct = s
        return self

    # reference accessor names (dataset.py:27-37, :78-86)
    def get_n_samples(self):
        return self.n_samples

    def get_n_features(self):
        return self.n_features

    def count_nonzero(self):
        return self.nnz

    def ref(self):
        return C.byref(self.struct)

    def col_norm_sq(self):
        out = torch.empty(self.n_features, dtype=torch.float64, device=self.device)
        _lib.check(_lib.load().sp_col_norm_sq(self.ref(), _ptr(out), _stream()))
        return out


def get_dataset(X, order="c", device=None):
    """Same call shape as the reference factory (dataset.py:119-134): order="fortran" builds
    what the column sweeps need (CSC + the CSR used for cache precompute), anything else the
    row layout only."""
    if order == "fortran":
        return DeviceDataset(X, need_csr=True, need_csc=True, device=device)
    return DeviceDataset(X, need_csr=True, need_csc=False, device=device)


def _pow2_floor(v):
    p = 1
    while p * 2 <= v:
        p *= 2
    return p


def choose_geometry(ds, solver, n_cta=None, threads=None):
    """Cluster width / CTA size for the sequential sweeps from the mean column length."""
    import os
    env_c = os.environ.get("SPARSEPOLY_B200_NCTA")
    env_t = os.environ.get("SPARSEPOLY_B200_THREADS")
    if n_cta is None and env_c:
        n_cta = int(env_c)
    if threads is None and env_t:
        threads = int(env_t)
    avg = ds.nnz / max(ds.n_features, 1)
    if n_cta is None:
        # widest cluster that still leaves ~16 nonzeros of a column per CTA (measured on B200:
        # the step time is flat in the geometry once every nonzero has its own thread)
        n_cta = _pow2_floor(max(1, min(16, int(avg // 16))))
    if threads is None:
        per_cta = avg / n_cta
        if solver == "pbcd":
            threads = 32 * max(1, min(8, int(np.ceil(per_cta / 4))))      # ~4 nonzero rows per warp
        else:
            threads = 32 * max(1, min(8, int(np.ceil(1.5 * per_cta / 32))))   # 1.5 slots per nonzero
    return int(n_cta), int(threads)


WINDOW_SIZES = (256, 192, 128, 96, 64, 48, 32, 24, 16, 12, 8, 4, 2, 1)
WINDOW_MAX = 256              # SP_WINDOW_MAX: per-position arrays of the pcd / cd_linear engine CTA
PBCD_WINDOW_MAX = 64          # per-position arrays and cold-sum ring of the pbcd engine CTA (pbcd_window.cu)


class WindowPlan:
    """struct sp_wplan: the window plan of the pipelined pcd / cd_linear sweep (csrc/wplan.cu,
    csrc/pcd_window.cu).  build() returns False when no window size fits (then the cluster sweep
    is used)."""

    def __init__(self, ds, rec_stride, window=None, horizon=None, min_window=8, pbcd_shape=None):
        import os
        self.ds = ds
        self.lib = _lib.load()
        self.pbcd_shape = pbcd_shape            # (degree, k): plan of the block sweep (pbcd_window.cu)
        if pbcd_shape is not None:
            self.slot_cap = min(8192, int(self.lib.sp_pbcd_wplan_slot_cap(int(pbcd_shape[0]), int(pbcd_shape[1]))))
        else:
            self.slot_cap = min(8192, int(self.lib.sp_wplan_slot_cap(int(rec_stride))))
        env_b = os.environ.get("SPARSEPOLY_B200_WINDOW")
        env_h = os.environ.get("SPARSEPOLY_B200_HORIZON")
        self.window = int(env_b) if (window is None and env_b) else window
        wmax = WINDOW_MAX if pbcd_shape is None else PBCD_WINDOW_MAX
        if self.window is not None and not 1 <= self.window <= wmax:
            raise ValueError(f"window plan: window={self.window} is outside 1..{wmax} for the "
                             f"{'pcd' if pbcd_shape is None else 'pbcd'} window sweep")
        self.horizon = int(env_h) if (horizon is None and env_h) else (0 if horizon is None else horizon)
        env_n = os.environ.get("SPARSEPOLY_B200_NEAR")
        self.near = int(env_n) if env_n else 1
        vec = 1
        if pbcd_shape is not None:
            self.near = 0                       # the block engine resolves every dependency in the workers
            vec = int(pbcd_shape[1])
        self.min_window = min_window
        self.max_hot_frac = 0.5
        dev, d = ds.device, ds.n_features
        self.pos = torch.empty(max(d, 1), dtype=torch.int32, device=dev)
        self.cflag = torch.empty(max(ds.nnz, 1), dtype=torch.int32, device=dev)
        self.hot_count = torch.zeros(max(d, 1), dtype=torch.int32, device=dev)
        self.ht_ptr = torch.zeros(d + 1, dtype=torch.int32, device=dev)
        self.res = torch.zeros(2 * max(d, 1) * vec, dtype=torch.float64, device=dev)
        n_base = 2 * max(d, 1) if pbcd_shape is None else int(self.lib.sp_pbcd_wplan_base_doubles())
        self.base = torch.zeros(n_base, dtype=torch.float64, device=dev)
        self.overflow = torch.zeros(1, dtype=torch.int32, device=dev)
        self.struct = None
        self.stats = {}

    def _candidates(self):
        if self.window is not None:
            return [int(self.window)]
        ds, H = self.ds, self.horizon
        col = ds.nnz / max(ds.n_features, 1)
        row = ds.nnz / max(ds.n_samples, 1)
        out = []
        for B in WINDOW_SIZES:
            if B < self.min_window:
                break
            if self.pbcd_shape is not None and B > 32:   # measured at C3: 16-32 positions per window is best
                continue
            if self.pbcd_shape is None and B > 96:       # measured at C2 (64 / 80 / 96 / 112 / 128 / 160): 96
                continue
            f = min(1.0, (2 * H + 1) * B * row / max(ds.n_features, 1))   # expected hot fraction
            if f <= self.max_hot_frac and 0.5 * B * col * f <= self.slot_cap:
                out.append(B)
        return out

    def _try(self, idx_feat, B):
        ds, lib, d = self.ds, self.lib, self.ds.n_features
        _lib.check(lib.sp_wplan_flag(ds.ref(), _ptr(idx_feat), B, self.horizon, _ptr(self.pos),
                                     _ptr(self.cflag), _ptr(self.hot_count), _stream()))
        self.ht_ptr[1:] = torch.cumsum(self.hot_count[:d], 0).to(torch.int32)
        n_hot = int(self.ht_ptr[d].item())
        if self.window is None and n_hot > self.max_hot_frac * max(ds.nnz, 1):
            return False
        n_windows = (d + B - 1) // B
        dev = ds.device
        self.h_sd = torch.empty(max(n_hot, 1), dtype=torch.int32, device=dev)
        self.h_x = torch.empty(max(n_hot, 1), dtype=torch.float64, device=dev)
        tmp_sd = torch.empty(max(n_hot, 1), dtype=torch.int32, device=dev)
        tmp_x = torch.empty(max(n_hot, 1), dtype=torch.float64, device=dev)
        self.ht_cls = torch.zeros(max(d, 1), dtype=torch.int32, device=dev)
        self.n_slots = torch.zeros(n_windows, dtype=torch.int32, device=dev)
        self.slot_row = torch.empty(n_windows * self.slot_cap, dtype=torch.int32, device=dev)
        self.sync = torch.zeros(4 * (n_windows + 2) + 2, dtype=torch.int32, device=dev)
        self.overflow.zero_()
        _lib.check(lib.sp_wplan_fill(ds.ref(), _ptr(idx_feat), B, self.slot_cap,
                                     2 if self.pbcd_shape is None else 3, self.near, _ptr(self.cflag),
                                     _ptr(self.ht_ptr), _ptr(tmp_sd), _ptr(tmp_x), _ptr(self.h_sd),
                                     _ptr(self.h_x), _ptr(self.ht_cls), _ptr(self.n_slots),
                                     _ptr(self.slot_row), _ptr(self.overflow), _stream()))
        if int(self.overflow.item()):
            # (what the failed window needed, for the error of a forced window)
            starts = torch.arange(0, d, B, device=dev)
            ends = torch.clamp(starts + B, max=d)
            self._overflow_need = (int(self.n_slots.max().item()),
                                   int((self.ht_ptr[ends] - self.ht_ptr[starts]).max().item()))
            return False
        s = _lib.SpWPlan()
        s.window, s.horizon, s.n_windows, s.slot_cap = B, self.horizon, n_windows, self.slot_cap
        s.near = self.near
        # SPARSEPOLY_B200_SPEC=0: never speculate on zero updates (debug / A-B measurements)
        s.flags = 1 if os.environ.get("SPARSEPOLY_B200_SPEC", "1") == "0" else 0
        s.flags |= (int(os.environ.get("SPARSEPOLY_B200_SPEC_DENOM", "0")) & 0xff) << 8   # debug: density threshold
        s.cflag, s.ht_ptr, s.ht_cls = self.cflag.data_ptr(), self.ht_ptr.data_ptr(), self.ht_cls.data_ptr()
        s.h_sd, s.h_x = self.h_sd.data_ptr(), self.h_x.data_ptr()
        s.n_slots, s.slot_row = self.n_slots.data_ptr(), self.slot_row.data_ptr()
        s.sync, s.res, s.base = self.sync.data_ptr(), self.res.data_ptr(), self.base.data_ptr()
        self.struct = s
        self.stats = dict(window=B, horizon=self.horizon, near=self.near, n_windows=n_windows, n_hot=n_hot,
                          hot_frac=n_hot / max(ds.nnz, 1), max_slots=int(self.n_slots.max().item()))
        return True

    def build(self, idx_feat):
        self.struct = None
        if self.ds.n_features == 0:
            return False
        near0 = self.near
        for B in self._candidates():
            # a position may hand at most 32 nonzeros to the chain warp: fall back to near=0 (every
            # hot nonzero goes through the worker warps) before shrinking the window
            for near in ((near0, 0) if near0 > 0 else (0,)):
                self.near = near
                if self._try(idx_feat, B):
                    self.near = near0
                    return True
        self.near = near0
        if self.window is not None:
            slots, hot = self._overflow_need
            ent_cap = (2 if self.pbcd_shape is None else 3) * self.slot_cap
            raise ValueError(f"window plan: window={self.window} horizon={self.horizon} does not fit "
                             f"{self.slot_cap} shared-memory slots: a window needs {slots} slots and "
                             f"{hot} hot nonzeros (at most {self.slot_cap} and {ent_cap})")
        return False


class SweepPlan:
    """Coordinate-order plan (struct sp_plan): per-position column slices of every CTA and the
    read-after-write hazard flags.  Rebuilt (cheaply, on device) whenever the order changes.

    sweep="window" (pcd / cd_linear only) additionally builds the WindowPlan of the pipelined
    sweep; "auto" uses it when the columns are sparse enough for it to fit, "cluster" never.
    Environment override: SPARSEPOLY_B200_SWEEP."""

    def __init__(self, ds, solver="pcd", n_cta=None, threads=None, rec_stride=None, sweep=None, pbcd_shape=None):
        import os
        self.ds = ds
        if sweep is None:
            sweep = os.environ.get("SPARSEPOLY_B200_SWEEP", "auto")
        if solver == "pcd" and rec_stride is None:
            sweep = "cluster"
        if solver == "pbcd" and (pbcd_shape is None or pbcd_shape[1] > 32):
            sweep = "cluster"
        self.sweep = sweep
        self.wplan = None
        if sweep in ("auto", "window"):
            self.wplan = WindowPlan(ds, rec_stride, min_window=8 if sweep == "auto" else 1,
                                    pbcd_shape=pbcd_shape if solver == "pbcd" else None)
            if self.wplan.slot_cap < 1:
                self.wplan = None
        if self.wplan is not None:
            if sweep == "window" and self.wplan.window is None:
                self.wplan.max_hot_frac = 2.0
        self.n_cta, self.threads = choose_geometry(ds, solver, n_cta, threads)
        self.idx_feat = torch.empty(max(ds.n_features, 1), dtype=torch.int32, device=ds.device)
        self._order_host = None
        self._cluster_ready = False
        s = _lib.SpPlan()
        s.n_cta, s.threads = self.n_cta, self.threads
        s.idx_feat = self.idx_feat.data_ptr()
        self.struct = s
        self.mode = "cluster"
        if self.wplan is None:
            self._ensure_cluster()

    def _ensure_cluster(self):
        """Buffers of the cluster sweep (allocated only when the window sweep is not used)."""
        if self._cluster_ready:
            return
        ds, dev = self.ds, self.ds.device
        d, C_ = ds.n_features, self.n_cta
        self.col_part = torch.empty(max(d * (C_ + 1), 1), dtype=torch.int32, device=dev)
        self.pos_ptr = torch.empty(max(d * (C_ + 1), 1), dtype=torch.int32, device=dev)
        self.flag_idx = torch.empty(max(ds.nnz, 1), dtype=torch.int32, device=dev)
        self.pos_conf = torch.zeros(max(d, 1), dtype=torch.int32, device=dev)
        _lib.check(_lib.load().sp_plan_partition(ds.ref(), C_, _ptr(self.col_part), _stream()))
        s = self.struct
        s.pos_ptr, s.flag_idx, s.pos_conf = (self.pos_ptr.data_ptr(), self.flag_idx.data_ptr(),
                                             self.pos_conf.data_ptr())
        self._cluster_ready = True

    def set_order(self, idx_feat_host):
        idx = np.ascontiguousarray(idx_feat_host, dtype=np.int32)
        if self._order_host is not None and np.array_equal(idx, self._order_host):
            return
        self._order_host = idx.copy()
        self.idx_feat[: idx.size].copy_(torch.from_numpy(idx))
        self.struct.win = None
        self.mode = "cluster"
        if self.wplan is not None and self.wplan.build(self.idx_feat):
            self.struct.win = C.pointer(self.wplan.struct)
            self.mode = "window"
            return
        self._ensure_cluster()
        _lib.check(_lib.load().sp_plan_order(self.ds.ref(), self.n_cta, _ptr(self.col_part),
                                             _ptr(self.idx_feat), _ptr(self.pos_ptr),
                                             _ptr(self.flag_idx), _ptr(self.pos_conf), _stream()))

    def ref(self):
        return C.byref(self.struct)
