#!/usr/bin/env python
"""bench.py -- headline benchmark of the sparsepoly B200 backend (contract in the task prompt).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--workload auto|psgd|pcd|pbcd|allsub|c1] [--scale S] [--dump-outputs DIR]

Workloads (BASELINE.json configs / SURVEY.md 8d):
  psgd   C5  FM-Clf degree=2 psgd squaredl12 logistic, Criteo-shaped d=1M 39 nnz/row k=32,
             sample-sharded, 6.25M rows per GPU (= n=50M at 8 GPUs)               [headline at every N]
  pcd    C2  FM-Clf degree=3 pcd omegati logistic, n=1M d=100k 50 nnz/row k=16
  pbcd   C3  FM-Reg degree=2 pbcd omegacs, n=1M d=100k 50 nnz/row k=32
  allsub C4  AllSubsets-Clf pcd omegati squared_hinge, n=500k d=20k 20 nnz/row k=16
  c1     C1  FM-Reg degree=2 pcd squaredl12, n=10k d=1k 50 nnz/row k=10 (the reference's CPU-runnable case)
A "step" is one epoch: for psgd one pass over the rank's 6.25M-row shard (244 minibatches of
batch_size="auto" samples per rank -- weak scaling: the global minibatch is auto x N), for the others one
sweep over all coordinates.  psgd is the path that shards (samples over the ranks, P over the ranks' HBM,
peer-memory exchange); pcd / pbcd are sequential in the coordinate order and stay on one GPU.
With --workload auto (default) the headline line is psgd; at N=1 the "also" list carries C2, C3, C4 and C1,
each with its own roofline / e2e / cpu_baseline; at N>1 it carries the strong-scaling psgd run (global
minibatch = auto, split over the ranks).
`--steps K` is the number of timed epochs of the headline workload (and of its e2e fit).  The "also" entries keep
their own fixed counts (3 epochs, 10 for C1, min(K, 10) for the strong-scaling run) so that the secondary lines
stay comparable whatever K is; each entry reports its own `steps`.

`--dump-outputs DIR` writes the model the headline workload's timed epochs computed (P_ and w_, as a caller of fit()
receives them) to DIR/<name>.npy in float64, at most 64 MB in all.  The inputs are seeded, so two builds of the
project can be compared output for output.

`--impl reference` times the reference algorithm on the host CPU (the pinned C oracle port of the numba
path, 1 core -- the reference is single threaded; the numba package itself cannot travel to the GPU box) on
a bounded sample of the same workload.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    "pcd": dict(tag="C2", n=1_000_000, d=100_000, r=50, seed=1, k=16, degree=3, clf=True,
                kw=dict(degree=3, loss="logistic", n_components=16, solver="pcd", regularizer="omegati",
                        alpha=1e-6, beta=1e-6, gamma=5e-10, mean=True, fit_linear=True,
                        fit_lower="explicit", shuffle=False, random_state=0, tol=-1.0)),
    "pbcd": dict(tag="C3", n=1_000_000, d=100_000, r=50, seed=2, k=32, degree=2, clf=False,
                 kw=dict(degree=2, n_components=32, solver="pbcd", regularizer="omegacs", alpha=1e-6,
                         beta=1e-6, gamma=1e-8, mean=True, fit_linear=True, fit_lower="explicit",
                         shuffle=False, random_state=0, tol=-1.0)),
    "allsub": dict(tag="C4", n=500_000, d=20_000, r=20, seed=3, k=16, degree=-1, clf=True,
                   kw=dict(loss="squared_hinge", n_components=16, solver="pcd", regularizer="omegati",
                           # OmegaTI for all-subsets multiplies gamma by prod_j (1 + |p_sj|) ~ e^160 at
                           # d=20k (reference omegati.py:19-34): only an absurdly small gamma leaves ~10 % of P_
                           beta=1e-6, gamma=1e-100, mean=True, shuffle=False, random_state=0, tol=-1.0)),
    "c1": dict(tag="C1", n=10_000, d=1_000, r=50, seed=0, k=10, degree=2, clf=False,
               kw=dict(degree=2, n_components=10, solver="pcd", regularizer="squaredl12", alpha=1e-3, beta=1e-3,
                       gamma=1e-4, mean=True, fit_linear=True, fit_lower="explicit", shuffle=False,
                       random_state=0, tol=-1.0)),
    "psgd": dict(tag="C5", n_per_gpu=6_250_000, d=1_000_000, r=39, seed=4, k=32, degree=2, clf=True,
                 kw=dict(degree=2, loss="logistic", n_components=32, solver="psgd",
                         # gamma: 20-30 % of P_ still nonzero after 5 epochs (1 220 updates), 6 % after the 26 of a default run
                         regularizer="squaredl12", alpha=1e-7, beta=1e-7, gamma=2e-8, fit_linear=True,
                         fit_lower="explicit", batch_size="auto", eta0=0.1, learning_rate="optimal",
                         power_t=1.0, shuffle=False, random_state=0, tol=-1.0, n_iter_no_change=10 ** 9)),
}


# --------------------------------------------------------------------------------- utilities
class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.gpu)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1])); smax.append(float(r[2]))
                for nm, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                pass
        out = {"sm_mhz": float(np.median(sm)) if sm else None,
               "sm_max_mhz": float(max(smax)) if smax else None, "reasons": sorted(reasons),
               "samples": len(sm)}
        if not sm:
            out["note"] = "timed region shorter than the 200 ms sampling period of nvidia-smi"
        return out


def profiled_traffic(kernel_key):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from the
    committed `ncu --set full` capture (profiles/traffic.json); None when there is no capture."""
    try:
        with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "traffic.json")) as f:
            return json.load(f).get(kernel_key, {}).get("dram_bytes_per_launch")
    except Exception:
        return None


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


ROWS_OVERRIDE = 0


def make_problem(name, scale=1.0, rank=0):
    """Synthetic inputs of the named config (host numpy / scipy)."""
    from sparsepoly_b200 import synth
    wl = WORKLOADS[name]
    if name == "psgd":
        n = max(1024, int((ROWS_OVERRIDE or wl["n_per_gpu"]) * scale))
        d = max(64, int(wl["d"] * scale))
        X = synth.criteo_like(n, d, wl["seed"] * 1000 + rank)
        # planted sparse degree-2 model on 10 % of the features (SURVEY.md 8d), CTR-like class balance;
        # the model is the same on every rank (seed without the rank), the noise is not
        y = synth.planted_fm_targets(X, wl["seed"], 99 + rank, positive_frac=0.25)
        return X, y
    n, d = max(256, int(wl["n"] * scale)), max(32, int(wl["d"] * scale))
    X = synth.uniform_sparse(n, d, wl["r"], wl["seed"] + 17 * rank)
    rng = np.random.RandomState(wl["seed"] + 100 + rank)
    # planted sparse linear + pairwise signal on 10% of the features (cheap host-side proxy for the
    # planted-model targets of SURVEY.md 8d; the timing does not depend on y)
    active = rng.choice(d, size=max(2, d // 10), replace=False)
    beta = np.zeros(d); beta[active] = rng.randn(active.size)
    s = X @ beta
    s = s + 0.5 * (s ** 2 - np.mean(s ** 2)) + 0.1 * np.std(s) * rng.randn(n)
    y = np.where(s > np.median(s), 1.0, -1.0) if wl["clf"] else (s / np.std(s))
    return X, y


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """Write every array as out_dir/<name>.npy in float64.  An array larger than its share of DUMP_BYTES is replaced
    by a fixed, seeded sample of its last (feature) axis: the same columns in every run with the same arguments."""
    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_BYTES // len(arrays)
    for name, a in arrays.items():
        a = np.ascontiguousarray(a, dtype=np.float64)
        if a.nbytes > share:
            keep = share // (a.nbytes // a.shape[-1])
            a = a[..., np.sort(np.random.RandomState(0).choice(a.shape[-1], keep, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def sweep_bytes(name, nnz, n, k, degree, fit_linear):
    """Algorithmic bytes of the SWEEP kernels in one epoch (SURVEY.md 8d byte model: column
    idx+val 12 B, A^1..A^(m-1) read+write 16(m-1) B, y_pred r/w 16 B, y 8 B per nonzero)."""
    lin = nnz * 36.0 if fit_linear else 0.0
    if name in ("pcd", "c1"):
        tot = lin
        for deg in range(2, degree + 1):
            tot += k * nnz * (12 + 16 * (deg - 1) + 24)
        return tot
    if name == "allsub":
        return k * nnz * (12 + 16 + 24)
    if name == "pbcd":
        return lin + nnz * (12 + 16 * k * (degree - 1) + 24)
    raise ValueError(name)


# --------------------------------------------------------------------------------- CPU arm
def cpu_reference_epoch_seconds(name, X, y, budget_s):
    """Time the reference algorithm (C oracle port, 1 host core -- the reference is single
    threaded) on a bounded sample and extrapolate to one full epoch of the workload.
    Sample = a leading slice of the columns (all rows), one component per order; CPU cost is
    linear in nnz x components.  Returns (seconds_per_epoch, description)."""
    from oracle import oracle as O
    import scipy.sparse as sp
    wl = WORKLOADS[name]
    kw = wl["kw"]
    n, d = X.shape
    k = wl["k"]
    # ~100 ns per nonzero-component-pass on one core: pick the column fraction for the budget
    passes = {"pcd": 1 + 2 * 5, "pbcd": 1 + 3 * 32 / 2.0, "allsub": 4, "c1": 1 + 5}[name]
    frac = min(1.0, budget_s / (X.nnz * passes * 60e-9))
    d_s = max(16, int(d * frac))
    Xs = sp.csc_matrix(X[:, :d_s])
    csc = O.to_csc(Xs)
    frac = Xs.nnz / X.nnz
    rng = np.random.RandomState(0)
    idx_feat = np.arange(d_s, dtype=np.int32)
    a_, b_, g_ = (kw.get("alpha", 1) * n, kw["beta"] * n, kw["gamma"] * n)
    loss = kw.get("loss", "squared")
    y_pred = np.zeros(n)
    t_total = 0.0
    if name in ("pcd", "allsub", "c1"):
        reg = O.Reg(kw["regularizer"], d_s, 1)
        lams = np.ones(1)
        idx_comp = np.zeros(1, dtype=np.int32)
        if name in ("pcd", "c1"):
            w = np.zeros(d_s)
            cns = O.col_norm_sq(Xs)
            t0 = time.perf_counter()
            O.cd_linear_epoch(w, csc, y, y_pred, cns, a_, loss, idx_feat)
            t_lin = time.perf_counter() - t0
            t_comp = 0.0
            reg.init_pcd(wl["degree"])
            for deg in range(2, wl["degree"] + 1):
                P = 0.01 * rng.randn(1, d_s)
                A = np.zeros((n, deg + 1))
                t0 = time.perf_counter()
                O.pcd_epoch(P, csc, y, y_pred, lams, deg, b_, g_, 1.0, reg, loss, A, idx_comp, idx_feat)
                t_comp += time.perf_counter() - t0
            t_total = (t_lin + k * t_comp) / frac
        else:
            reg.init_pcd(-1)
            P = 0.01 * rng.randn(1, d_s)
            A = np.ones(n)
            y_pred = np.ones(n)
            t0 = time.perf_counter()
            O.pcd_all_epoch(P, csc, y, y_pred, lams, b_, g_, kw.get("eta0", 0.1), reg, loss, A, idx_comp, idx_feat)
            t_total = k * (time.perf_counter() - t0) / frac
        desc = (f"C oracle port of the numba path, 1 core: {d_s}/{d} leading columns ({frac:.3%} of nnz), "
                f"all {n} rows, 1 of {k} components per order, extrapolated linearly")
    else:  # pbcd
        kk = k
        reg = O.Reg(kw["regularizer"], d_s, kk)
        reg.init_pbcd(wl["degree"])
        w = np.zeros(d_s)
        cns = O.col_norm_sq(Xs)
        t0 = time.perf_counter()
        O.cd_linear_epoch(w, csc, y, y_pred, cns, a_, loss, idx_feat)
        P = np.ascontiguousarray(0.01 * rng.randn(d_s, kk))
        A = np.zeros((n, wl["degree"] + 1, kk))
        dA = np.zeros((n, wl["degree"], kk))
        O.pbcd_epoch(P, csc, y, y_pred, np.ones(kk), wl["degree"], b_, g_, 1.0, reg, loss, A, dA, idx_feat)
        t_total = (time.perf_counter() - t0) / frac
        desc = (f"C oracle port of the numba path, 1 core: {d_s}/{d} leading columns ({frac:.3%} of nnz), "
                f"all {n} rows, all {kk} components, extrapolated linearly")
    return t_total, desc


_REAL_REF = {}


def real_reference_psgd_samples_per_s(X, y, budget_s):
    """The UNMODIFIED reference (numba) on the host: oracle/_ref/reference_pkg is a git-ignored copy staged in the
    build container (scripts/run_reference_suite.py --stage); returns None when it (or numba) is not there."""
    pkg = os.path.join(ROOT, "oracle", "_ref", "reference_pkg")
    if not os.path.isdir(os.path.join(pkg, "sparsepoly")):
        return None
    try:
        if "cls" not in _REAL_REF:
            sys.path.insert(0, pkg)
            os.environ.setdefault("NUMBA_CACHE_DIR", "/tmp/numba_cache")
            import sparsepoly as ref_pkg
            _REAL_REF["cls"] = ref_pkg.SparseFactorizationMachineClassifier
            sys.path.remove(pkg)
    except Exception as e:                                   # numba missing / import error: fall back to the port
        _REAL_REF["error"] = repr(e)
        return None
    import warnings
    wl = WORKLOADS["psgd"]
    kw = dict(wl["kw"])
    n, d = X.shape
    batch = int(n * d / X.nnz)
    kw["batch_size"] = batch
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        if not _REAL_REF.get("warm"):                        # JIT compilation of this specialisation (not timed)
            _REAL_REF["cls"](max_iter=1, **dict(kw, batch_size=64)).fit(X[:256], y[:256])
            _REAL_REF["warm"] = True
        # ~3 s per minibatch on one core (25 641 samples + dense update / prox of 32 M entries)
        nb = max(1, int(budget_s / 3.0))
        ns = min(n, nb * batch)
        t0 = time.perf_counter()
        _REAL_REF["cls"](max_iter=1, **kw).fit(X[:ns], y[:ns])
        dt = time.perf_counter() - t0
    return ns / dt, (f"the unmodified reference (numba {__import__('numba').__version__}, 1 core): fit(max_iter=1) on the first "
                     f"{ns} samples = {ns // batch} minibatches of {batch} at full d={d}, k={wl['k']} (includes its host-side "
                     f"P_ initialisation and CSR conversion)")


def cpu_reference_psgd_samples_per_s(X, y, budget_s):
    from oracle import oracle as O
    wl = WORKLOADS["psgd"]
    kw = wl["kw"]
    n, d = X.shape
    k = wl["k"]
    batch = int(n * d / X.nnz)
    # ~2 us/sample sparse part + dense update+prox ~ 3*d*k*8 B at ~5 GB/s effective per minibatch
    per_batch = batch * 3e-6 + d * k * 25e-9
    nb = max(1, int(budget_s / per_batch))
    ns = min(n, nb * batch)
    Xs = X[:ns]
    csr = O.to_csr(Xs)
    reg = O.Reg(kw["regularizer"], d, k)
    P = np.ascontiguousarray(0.01 * np.random.RandomState(0).randn(1, d, k))
    w = np.zeros(d)
    gP, gw = np.zeros_like(P), np.zeros(d)
    idx = np.arange(ns, dtype=np.int32)
    t0 = time.perf_counter()
    O.psgd_epoch(csr, y[:ns], P, w, np.ones(k), 2, kw["alpha"], kw["beta"], kw["gamma"], reg, kw["loss"],
                 gP, gw, idx, True, kw["eta0"], 1, kw["power_t"], batch, 1)
    dt = time.perf_counter() - t0
    return ns / dt, (f"C oracle port of the numba path, 1 core: first {ns} samples = {ns // batch} minibatches "
                     f"of {batch} at full d={d}, k={k}")


def sweep_config(name, args, X, world):
    """`config` of a pcd / pbcd line: identical in both arms (ours / reference)."""
    wl = WORKLOADS[name]
    n, d = X.shape
    return {"workload": f"{wl['tag']} {name}: " + json.dumps(wl["kw"]),
            "n_samples": n, "n_features": d, "nnz": int(X.nnz), "scale": args.scale,
            "l2": "inputs_exceed_l2 (CSC+CSR+records >> 126 MB)" if X.nnz * 24 > 2e8 else "inputs fit L2",
            "parallelism": "single GPU" if world == 1 else f"{world} independent replicas (pcd/pbcd do not shard)"}


# --------------------------------------------------------------------------------- GPU arm
def run_sweep_workload(name, args, rank, world, local, dump_dir=None):
    import torch
    import sparsepoly_b200 as S
    from sparsepoly_b200 import _lib
    wl = WORKLOADS[name]
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    X, y = make_problem(name, args.scale, rank)
    n, d = X.shape
    kw = dict(wl["kw"], max_iter=args.steps)
    if args.gamma is not None:
        kw["gamma"] = args.gamma
    if name == "allsub":
        cls = S.SparseAllSubsetsClassifier
    else:
        cls = S.SparseFactorizationMachineClassifier if wl["clf"] else S.SparseFactorizationMachineRegressor
    lib = _lib.load()

    # ---- device-resident timing: inputs in HBM, W warm-up + K timed epochs, CUDA events
    est = cls(**kw)
    Xc, yc = est._check_X_y(X, y)
    from sklearn.utils import check_random_state
    rng = check_random_state(kw["random_state"])
    lib.sp_set_device(local)
    if name == "allsub":
        est.P_ = 0.01 * rng.randn(est.n_components, Xc.shape[1])
        est.lams_ = np.ones(est.n_components)
        setup = est._setup
    else:
        Xc = est._augment(Xc)
        est.w_ = np.zeros(Xc.shape[1])
        n_orders = est.degree - 1 if est.fit_lower == "explicit" else 1
        est.P_ = 0.01 * rng.randn(n_orders, est.n_components, Xc.shape[1])
        est.lams_ = np.ones(est.n_components)
        setup = est._pcd_setup if name in ("pcd", "c1") else est._pbcd_setup
    epoch, sync = setup(Xc, np.ascontiguousarray(yc, dtype=np.float64), rng, dev)
    first_epochs = []                                  # the dense regime: P_ starts fully dense (0.01 * randn)
    for _ in range(args.warmup):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        epoch(read_back=False)
        e1.record()
        torch.cuda.synchronize()
        first_epochs.append(e0.elapsed_time(e1) / 1e3)
    torch.cuda.synchronize()
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
    lib.sp_profile_enable(1)
    import ctypes as C
    _z = (C.c_ulonglong * 2)()
    lib.sp_wspec_read(_z)                       # reset the speculation counters
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    ev0.record()
    for _ in range(args.steps):
        epoch(read_back=False)
    ev1.record()
    torch.cuda.synchronize()
    clocks = sampler.stop() if rank == 0 else None
    ms_total = ev0.elapsed_time(ev1)
    import ctypes as C
    ms = (C.c_double * 8)()
    cnt = (C.c_longlong * 8)()
    lib.sp_profile_collect(ms, cnt)
    lib.sp_profile_enable(0)
    wspec = (C.c_ulonglong * 2)()
    lib.sp_wspec_read(wspec)
    sync()
    if dump_dir is not None and rank == 0:
        dump_outputs(dump_dir, {"P_": est.P_, **({"w_": est.w_} if hasattr(est, "w_") else {})})
    nz_frac = float(np.mean(est.P_ != 0))
    nz_by_order = ([float(np.mean(est.P_[o] != 0)) for o in range(est.P_.shape[0])]
                   if est.P_.ndim == 3 else [nz_frac])
    if world > 1:
        t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t.item())
    sec_per_epoch = ms_total / 1e3 / args.steps
    cls_id = 3 if name == "pbcd" else 2
    sweep_ms, sweep_n = float(ms[cls_id]) + (float(ms[2]) if name == "pbcd" else 0.0), int(cnt[cls_id])
    alg_bytes = sweep_bytes(name, X.nnz, n, wl["k"], wl["degree"], True) * args.steps
    peak, peak_src = measured_peak()
    achieved = alg_bytes / (sweep_ms / 1e3) / 1e9 if sweep_ms > 0 else 0.0
    coords = (d * (1 + wl["k"] * (wl["degree"] - 1))) if name in ("pcd", "c1") else (d * wl["k"] if name == "allsub" else 2 * d)
    result = {
        "value": sec_per_epoch, "ms_per_step": sec_per_epoch * 1e3,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "traffic": None, "peak_source": peak_src,
                     "kernel": "sweep_kernel (pcd.cu)" if name in ("pcd", "c1", "allsub") else "pbcd_sweep_kernel (pbcd.cu)",
                     "kernel_ms_per_step": sweep_ms / args.steps,
                     "kernel_share_of_step": sweep_ms / ms_total if ms_total else None,
                     "algorithmic_bytes_per_step": alg_bytes / args.steps,
                     "sequential_steps_per_epoch": coords,
                     "us_per_sequential_step": sweep_ms * 1e3 / args.steps / coords},
        "gpu_launches": int(sum(cnt)),
        "kernel_ms": {"rows": ms[0], "regcache": ms[1], "sweep_pcd": ms[2], "sweep_pbcd": ms[3]},
        "clocks": clocks, "p_nonzero_frac": nz_frac, "p_nonzero_frac_by_order": nz_by_order,
        "dense_regime_epochs_s": first_epochs,
        "dense_regime_note": "epochs 1..warmup from the dense random start (every coordinate moves), device-timed one by "
                             "one; `value` is the steady state after them",
        "zero_update_speculation": {"positions": int(wspec[0]), "rejected": int(wspec[1]),
                                    "note": "window-sweep positions evaluated without per-record waits (pcd_window.cu)"},
        "geometry": ({"sweep": "window", **est._dev_state["plan"].wplan.stats}
                     if getattr(est._dev_state["plan"], "mode", "cluster") == "window" else
                     {"sweep": "cluster", "n_cta": est._dev_state["plan"].n_cta,
                      "threads": est._dev_state["plan"].threads}),
    }
    if result["geometry"]["sweep"] == "window" and name == "pbcd":
        result["roofline"]["kernel"] = "pbcd_wsweep_kernel (pbcd_window.cu)"
    if result["geometry"]["sweep"] == "window" and name in ("pcd", "allsub", "c1"):
        result["roofline"]["kernel"] = "wsweep_kernel (pcd_window.cu)"
        if name == "pcd" and args.scale == 1.0:
            result["roofline"]["traffic"] = profiled_traffic("wsweep_kernel")
        result["roofline"]["algorithmic_bytes_per_launch"] = alg_bytes / args.steps / max(1, sweep_n // args.steps)
    del est, epoch, sync
    torch.cuda.empty_cache()

    # ---- end to end through the public API: host buffers in, fitted host arrays out
    est2 = cls(**kw)
    import warnings
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        est2.fit(X, y)
    torch.cuda.synchronize()
    e2e_s = (time.perf_counter() - t0) / args.steps
    if world > 1:
        t = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    if rank == 0:
        # objective the fit reached (device evaluator, csrc/objective.cu; outside every timed region)
        from sparsepoly_b200.objective import objective
        result["objective"] = objective(est2, X, y)
    result["e2e"] = {"value": e2e_s, "unit": "s/epoch", "h2d_bytes_per_step": int(est2._h2d_bytes / args.steps),
                     "d2h_bytes_per_step": int((est2.P_.nbytes + getattr(est2, "w_", np.zeros(0)).nbytes) / args.steps + 8),
                     "note": f"fit(X_host, y_host) wall clock / {args.steps} epochs: host CSR->CSC, H2D, epochs, D2H"}
    if rank == 0 and not args.no_cpu:
        t_cpu, desc = cpu_reference_epoch_seconds(name, X, y, args.cpu_budget)
        result["cpu_baseline"] = {"value": t_cpu, "unit": "s/epoch", "cores": 1, "kind": "port", "sample": desc}
    result["config"] = sweep_config(name, args, X, world)
    return result


def psgd_config(args, world, batch_mode):
    """`config` of the psgd line: identical in both arms (ours / reference)."""
    wl = WORKLOADS["psgd"]
    n = max(1024, int((args.rows_per_gpu or wl["n_per_gpu"]) * args.scale))
    d = max(64, int(wl["d"] * args.scale))
    return {"workload": "C5 psgd: " + json.dumps(wl["kw"]), "rows_per_gpu": n, "n_features": d,
            "nnz_per_row": wl["r"], "scale": args.scale, "n_gpus": world,
            "batch": ("weak: global minibatch = batch_size('auto') x n_gpus, every rank contributes one auto-sized batch"
                      if batch_mode == "weak" else "strong: global minibatch = batch_size('auto'), split over the ranks"),
            "l2": "inputs_exceed_l2 (P is 256 MB, X 2.9 GB per GPU)" if d * wl["k"] * 8 > 1.3e8 else "P fits L2",
            "parallelism": ("single GPU" if world == 1 else
                            f"{world} ranks: samples sharded, P sharded by rows over the ranks' HBM, peer-memory "
                            f"pull / push / owner-update per minibatch (no NCCL on the data path)")}


def run_psgd_workload(args, rank, world, local, batch_mode="weak", dump_dir=None):
    """C5: step = one epoch over the rank's shard.  Device-timed value through the estimator's own epoch
    function with X / y / plan resident; e2e = fit(X_host, y_host) wall clock (H2D of X, plan, epochs, D2H)."""
    import ctypes as C
    import warnings
    import torch
    import sparsepoly_b200 as S
    from sklearn.utils import check_random_state
    from sparsepoly_b200 import _lib, distributed
    wl = WORKLOADS["psgd"]
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    lib = _lib.load()
    lib.sp_set_device(local)
    group = None
    if world > 1:
        import torch.distributed as dist
        group = distributed.enable_sharding()
    global ROWS_OVERRIDE
    ROWS_OVERRIDE = args.rows_per_gpu
    t_gen = time.perf_counter()
    X, y = make_problem("psgd", args.scale, rank)
    t_gen = time.perf_counter() - t_gen
    n, d = X.shape
    k, r = wl["k"], wl["r"]
    batch_auto = int(n * d / X.nnz)                   # batch_size="auto" = d / nnz_row (independent of n)
    kw = dict(wl["kw"])
    if args.gamma is not None:
        kw["gamma"] = args.gamma
    kw["batch_size"] = batch_auto * world if batch_mode == "weak" else batch_auto
    b_loc = max(1, kw["batch_size"] // world)
    est = S.SparseFactorizationMachineClassifier(max_iter=args.steps, **kw)
    Xc, yc = est._check_X_y(X, y)
    rng = check_random_state(kw["random_state"])
    est.w_ = np.zeros(d)
    est.P_ = 0.01 * rng.randn(1, k, d)
    est.lams_ = np.ones(k)
    est.it_ = 1
    t_setup = time.perf_counter()
    epoch, sync, close = est._psgd_setup(Xc, np.ascontiguousarray(yc, dtype=np.float64), rng, dev)
    torch.cuda.synchronize()
    t_setup = time.perf_counter() - t_setup
    n_mb = est._psgd_stats["minibatches"]
    for _ in range(args.warmup):
        epoch(read_back=False)
    torch.cuda.synchronize()
    if group is not None:
        dist.barrier()
    # timed region: K epochs as a user runs them (no per-kernel events: the ~10 event records per minibatch
    # of the profiled pass below cost ~7 % at N=1)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    ev0.record()
    for _ in range(args.steps):
        epoch(read_back=False)
    ev1.record()
    torch.cuda.synchronize()
    clocks = sampler.stop() if rank == 0 else None
    ms_total = ev0.elapsed_time(ev1)
    if dump_dir is not None:
        # the model after the last timed epoch, as a fit() callback would see it.  On the planned path sync() folds
        # the lazy scales into the stored model, so the epochs after this point (profiled pass, final read-back) can
        # differ in the last bits from a run without --dump-outputs; the timed value above is not affected.
        sync()
        if rank == 0:
            dump_outputs(dump_dir, {"P_": est.P_, "w_": est.w_})
    # profiled pass: the same K epochs again with a CUDA-event pair around every kernel class (sp_profile_*, on the
    # launching streams): the kernel durations of the roofline and the per-class figures
    if group is not None:
        dist.barrier()
    lib.sp_profile_enable(1)
    evp0, evp1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    evp0.record()
    for _ in range(args.steps):
        epoch(read_back=False)
    evp1.record()
    torch.cuda.synchronize()
    ms_prof_total = evp0.elapsed_time(evp1)
    ms = (C.c_double * 8)()
    cnt = (C.c_longlong * 8)()
    lib.sp_profile_collect(ms, cnt)
    lib.sp_profile_enable(0)
    last_loss = epoch()                              # one more epoch, read back: the metric a user sees
    sync()
    nz_frac = float(np.mean(est.P_ != 0))
    close()
    selection = est._psgd_stats.get("selection")
    if group is not None:
        t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t.item())
    samples = args.steps * n * world
    value = samples / (ms_total / 1e3)
    # SURVEY.md 8d byte model: per sample (rows pass: CSR + P gather + w; column pass: grad_P / grad_w
    # read-modify-write) and per minibatch (5 dense sweeps of P / grad_P + 4 of w / grad_w)
    rows_bytes = r * 12 + r * k * 8 + r * 8 + 8
    cols_bytes = 2 * r * k * 8 + 2 * r * 8
    dense_bytes = 5 * d * k * 8 + 4 * d * 8
    peak, peak_src = measured_peak()
    n_launch = args.steps * n_mb
    klass = {"psgd_rows_kernel": (float(ms[4]), rows_bytes * b_loc),
             "psgd_cols_{long,combine,single,short}_kernel": (float(ms[5]), cols_bytes * b_loc),
             "psgd_stats_kernel + psgd_solve_kernel": (float(ms[6]) + float(ms[7]), dense_bytes)}
    dom = max(klass, key=lambda q: klass[q][0])
    dom_ms, dom_bytes = klass[dom]
    achieved = dom_bytes * n_launch / (dom_ms / 1e3) / 1e9 if dom_ms > 0 else 0.0
    step_bytes = (rows_bytes + cols_bytes) * n + dense_bytes * n_mb         # one epoch of one rank
    result = {
        "value": value, "ms_per_step": ms_total / args.steps,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": profiled_traffic(dom.split(" ")[0]), "peak_source": peak_src, "kernel": dom + " (psgd_plan.cu)",
                     "kernel_ms_per_launch": dom_ms / max(n_launch, 1),
                     "kernel_share_of_step": dom_ms / ms_prof_total if ms_prof_total else None,
                     "kernel_times_from": "a second pass of the same K epochs with per-class CUDA-event pairs "
                                          f"({ms_prof_total / args.steps:.3f} ms per epoch with the events; the timed "
                                          "region itself carries none)",
                     "algorithmic_bytes_per_launch": dom_bytes,
                     "byte_model": "SURVEY.md 8d per-unit figures x units per launch: rows 10.8 KB/sample, column pass "
                                   "20.6 KB/sample, dense sweeps 1.31 GB/minibatch; the planned path never makes the dense "
                                   "sweeps (touched rows only + one read-only statistics pass), so fractions above 1 are "
                                   "work avoided, not bandwidth",
                     "per_kernel": {q: {"ms_per_launch": v[0] / max(n_launch, 1), "algorithmic_bytes_per_launch": v[1],
                                        "gbs": v[1] * n_launch / (v[0] / 1e3) / 1e9 if v[0] > 0 else None} for q, v in klass.items()},
                     "whole_step_gbs_per_gpu": step_bytes * args.steps / (ms_total / 1e3) / 1e9,
                     "whole_step_frac": step_bytes * args.steps / (ms_total / 1e3) / 1e9 / peak},
        "gpu_launches": int(args.steps * (n_mb * (5 if kw["regularizer"] == "squaredl12" else 4) + 2)
                            + (args.steps * n_mb * 6 if world > 1 else 0)),     # (timed region; the profiled pass repeats it)
        "stats_us_per_minibatch": 1e3 * float(ms[6]) / max(n_launch, 1), "solve_us_per_minibatch": 1e3 * float(ms[7]) / max(n_launch, 1),
        "exchange_us_per_minibatch": ({"pull": 1e3 * float(ms[0]) / max(n_launch, 1), "inbox_barrier": 1e3 * float(ms[1]) / max(n_launch, 1),
                                       "owner_update": 1e3 * float(ms[2]) / max(n_launch, 1)} if world > 1 else None),
        "exchange_note": "sharded runs: peer-memory pull of the touched rows, flag barrier after the pushes, owner-side update (CUDA events)",
        "clocks": clocks, "p_nonzero_frac": nz_frac, "mean_loss_after": last_loss,
        "details": {"minibatches_per_epoch": n_mb, "batch_local": b_loc, "global_batch": b_loc * world,
                    "batch_size_auto": batch_auto, "columns_per_minibatch": est._psgd_stats["columns_per_minibatch"],
                    "plan_bytes": est._psgd_stats["plan_bytes"], "data_generation_s": t_gen, "setup_s": t_setup,
                    "setup_seconds": est._psgd_stats.get("setup_seconds"), "squaredl12_selection": selection},
    }
    del est, epoch, sync, close
    torch.cuda.empty_cache()
    # ---- end to end through the public API: host buffers in, fitted host arrays out
    e_epochs = max(1, args.steps)                     # the same number of steps as the device-timed region
    est2 = S.SparseFactorizationMachineClassifier(max_iter=e_epochs, **kw)
    torch.cuda.synchronize()
    if group is not None:
        dist.barrier()
    t0 = time.perf_counter()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        est2.fit(X, y)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    if group is not None:
        t = torch.tensor([dt], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dt = float(t.item())
    result["e2e"] = {"value": e_epochs * n * world / dt, "unit": "samples/s",
                     "h2d_bytes_per_step": int(est2._h2d_bytes / e_epochs),
                     "d2h_bytes_per_step": int((est2.P_.nbytes + est2.w_.nbytes) / e_epochs + 8),
                     "note": f"fit(X_host, y_host) wall clock over {e_epochs} epochs per rank: H2D of the CSR shard, batch-CSC "
                             f"plan (device sorts), epochs (loss read back each), D2H of P_ / w_"}
    if group is not None:
        distributed.disable_sharding()
    if rank == 0 and not args.no_cpu:
        v, desc = cpu_reference_psgd_samples_per_s(X, y, args.cpu_budget)
        result["cpu_baseline"] = {"value": v, "unit": "samples/s", "cores": 1, "kind": "port", "sample": desc}
    result["config"] = psgd_config(args, world, batch_mode)
    return result


def run_predict_workload(args, rank, world, local):
    """Batch prediction (base.py:52-100 -> kernels.poly_predict) of a C5-shaped model, samples sharded over the ranks,
    no collective on the compute path: device-timed sp_predict on resident shards + e2e decision_function(X_host)."""
    import torch
    import sparsepoly_b200 as S
    from sparsepoly_b200 import _lib, solvers
    from sparsepoly_b200.dataset import DeviceDataset
    wl = WORKLOADS["psgd"]
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    _lib.load().sp_set_device(local)
    global ROWS_OVERRIDE
    ROWS_OVERRIDE = min(args.rows_per_gpu or 2_000_000, 2_000_000)
    X, _ = make_problem("psgd", args.scale, rank)
    ROWS_OVERRIDE = args.rows_per_gpu
    n, d = X.shape
    k, r = wl["k"], wl["r"]
    rng = np.random.RandomState(0)
    est = S.SparseFactorizationMachineClassifier(**wl["kw"])
    est.P_ = 0.01 * rng.randn(1, k, d) * (rng.rand(1, k, d) < 0.1)        # a sparse fitted model (10 % nonzero)
    est.w_ = 0.01 * rng.randn(d)
    est.lams_ = np.ones(k)
    ds = DeviceDataset(X, need_csr=True, need_csc=False, device=dev, hot_features=False)
    P_dk = solvers.transpose(torch.from_numpy(est.P_[0]).to(dev))
    w = torch.from_numpy(est.w_).to(dev)
    lams = torch.ones(k, dtype=torch.float64, device=dev)
    out = torch.zeros(n, dtype=torch.float64, device=dev)
    for _ in range(3):
        solvers.poly_predict(ds, P_dk, lams, 2, w=w, out=out)
    torch.cuda.synchronize()
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
    reps = 10
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(reps):
        solvers.poly_predict(ds, P_dk, lams, 2, w=w, out=out)
    ev1.record()
    torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1)
    t0 = time.perf_counter()
    pred = est.decision_function(X)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([ms, dt], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, dt = float(t[0].item()), float(t[1].item())
    per_sample = r * 12 + r * k * 8 + r * 8 + 8                     # SURVEY.md 8d: 10.8 KB / sample
    peak, peak_src = measured_peak()
    value = reps * n * world / (ms / 1e3)
    gbs = per_sample * reps * n / (ms / 1e3) / 1e9
    return {"metric": "predict_samples_per_second", "value": value, "unit": "samples/s", "n_gpus": world, "steps": reps,
            "warmup": 3, "ms_per_step": ms / reps, "higher_is_better": True, "scaling": "weak", "dtype": "f64",
            "data": "synthetic",
            "roofline": {"bound": "hbm", "achieved": gbs, "peak": peak, "unit": "GB/s", "frac": gbs / peak, "traffic": None,
                         "peak_source": peak_src, "kernel": "rows_all_kernel (rows.cu)",
                         "algorithmic_bytes_per_launch": per_sample * n},
            "e2e": {"value": n * world / dt, "unit": "samples/s", "h2d_bytes_per_step": int(X.nnz * 12 + (n + 1) * 4 + est.P_.nbytes + est.w_.nbytes),
                    "d2h_bytes_per_step": int(pred.nbytes),
                    "note": "decision_function(X_host) wall clock per rank: H2D of the CSR shard and the model, kernel, D2H of the scores"},
            "gpu_launches": reps + 3,
            "config": {"workload": "C5-shaped batch prediction: degree=2, k=32, d=1M, 39 nnz/row, model 10 % nonzero",
                       "rows_per_gpu": n, "parallelism": "single GPU" if world == 1 else f"{world} ranks: samples sharded, model replicated, no collective"}}


def run_reference(args, rank, world):
    if rank != 0:
        return None
    name = args.workload
    global ROWS_OVERRIDE
    if name == "psgd":
        ROWS_OVERRIDE = args.rows_per_gpu or 1_000_000      # (the bounded sample only ever reads the leading rows)
    X, y = make_problem(name, args.scale, 0)
    per_step_budget = max(2.0, min(30.0, 150.0 / max(1, args.steps + args.warmup)))
    vals = []
    desc = ""
    t_run0 = time.perf_counter()
    kind = "port"
    for s in range(args.warmup + args.steps):
        if name == "psgd":
            real = real_reference_psgd_samples_per_s(X, y, per_step_budget)
            if real is not None:
                (v, desc), kind = real, "reference"
            else:
                v, desc = cpu_reference_psgd_samples_per_s(X, y, per_step_budget)
        else:
            v, desc = cpu_reference_epoch_seconds(name, X, y, per_step_budget)
        if s >= args.warmup:
            vals.append(v)
    wall = time.perf_counter() - t_run0
    value = float(np.mean(vals))
    unit = "samples/s" if name == "psgd" else "s/epoch"
    return {"impl": "reference", "metric": metric_name(name), "value": value, "unit": unit,
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": wall * 1e3 / max(1, args.steps + args.warmup),
            "higher_is_better": name == "psgd", "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": psgd_config(args, args.gpus, "weak") if name == "psgd" else sweep_config(name, args, X, 1),
            "cpu_baseline": {"value": value, "unit": unit, "cores": 1, "kind": kind, "sample": desc},
            "e2e": {"value": value, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}


def metric_name(name):
    return {"pcd": "pcd_epoch_seconds", "pbcd": "pbcd_epoch_seconds", "allsub": "pcd_allsubsets_epoch_seconds",
            "c1": "pcd_epoch_seconds", "psgd": "psgd_samples_per_second"}[name]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10, help="timed epochs of the headline workload")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="auto", choices=["auto", "pcd", "pbcd", "allsub", "c1", "psgd"])
    ap.add_argument("--scale", type=float, default=1.0, help="shrink n and d (debug only)")
    ap.add_argument("--cpu-budget", type=float, default=10.0)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--rows-per-gpu", type=int, default=0, help="psgd: override the shard size (debug)")
    ap.add_argument("--psgd-batch", default="weak", choices=["weak", "strong"],
                    help="psgd global minibatch: 'weak' (auto x n_gpus: per-GPU work fixed) or 'strong' (auto, split over the ranks)")
    ap.add_argument("--no-also", action="store_true", help="skip the secondary workloads")
    ap.add_argument("--gamma", type=float, default=None, help="override the workload's gamma (debug: other sparsity regimes)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write P_ / w_ as the headline workload's timed epochs left them to DIR/<name>.npy (float64, <= 64 MB)")
    args = ap.parse_args()
    rank, world, local = dist_env()
    global ROWS_OVERRIDE
    ROWS_OVERRIDE = args.rows_per_gpu
    auto = args.workload == "auto"
    if auto:
        args.workload = "psgd"
    args.warmup = max(3, args.warmup) if args.impl == "ours" else args.warmup

    if args.impl == "reference":
        out = run_reference(args, rank, world)
        if out is not None:
            print(json.dumps(out))
        return

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    name = args.workload
    if name == "psgd":
        res = run_psgd_workload(args, rank, world, local, args.psgd_batch, args.dump_outputs)
    else:
        res = run_sweep_workload(name, args, rank, world, local, args.dump_outputs)
    also = []
    if auto and not args.no_also:
        import copy
        if world == 1:
            # the sequential solvers (north_star: pcd / pbcd epoch time at 1 GPU), each with its CPU baseline
            for nm in ("pcd", "pbcd", "allsub", "c1"):
                a3 = copy.copy(args)
                a3.steps, a3.warmup = (3, 3) if nm != "c1" else (10, 3)
                a3.cpu_budget = min(args.cpu_budget, 8.0)
                r3 = run_sweep_workload(nm, a3, rank, world, local)
                r3.update(metric=metric_name(nm), unit="s/epoch", n_gpus=1, steps=a3.steps, warmup=a3.warmup,
                          higher_is_better=False, dtype="f64", data="synthetic")
                also.append(r3)
        else:
            a2 = copy.copy(args)
            a2.no_cpu = True
            a2.steps, a2.warmup = min(args.steps, 10), 3
            r2 = run_psgd_workload(a2, rank, world, local, "strong")
            r2.update(metric=metric_name("psgd"), unit="samples/s", n_gpus=world, steps=a2.steps, warmup=a2.warmup,
                      higher_is_better=True, scaling="strong", dtype="f64", data="synthetic")
            also.append(r2)
        also.append(run_predict_workload(args, rank, world, local))
    if rank == 0:
        line = {"metric": metric_name(name), "value": res.pop("value"),
                "unit": "samples/s" if name == "psgd" else "s/epoch", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": res.pop("ms_per_step"),
                "higher_is_better": name == "psgd",
                "scaling": "weak" if not (name == "psgd" and args.psgd_batch == "strong") else "strong",
                "vs_baseline": None, "dtype": "f64", "data": "synthetic"}
        line.update(res)
        if also:
            line["also"] = also
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
