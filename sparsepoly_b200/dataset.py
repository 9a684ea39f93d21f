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
        if need_csr:
            self.csr = tuple(_h2d(a, self.device, pin) for a in host_csr(X))
            self.h2d_bytes += sum(t.numel() * t.element_size() for t in self.csr)
        if need_csc:
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
