"""fit_many against the sequential fit loop; writes fit_many_bench.json (fit_many_pbcd_bench.json with
--solver pbcd) into OUTDIR.

    python scripts/fit_many_bench.py OUTDIR [--solver pcd|pbcd] [--epochs-a 20] [--epochs-bc 5]

pcd: (a) the reference notebook's grid: n=200, d=100, k=30, degree 2, dense, {l1, squaredl12, omegati} x 8 gamma
    x 4 beta = 96 models;  (b) the C1 shape: synth.uniform_sparse(10000, 1000, 50, 0), k=10, squaredl12,
    16 gamma values;  (c) one-vs-rest, 10 classes on (b)'s X.
pbcd: (a) the notebook grid with {l21, squaredl21, omegacs};  (b) the C1 shape with l21, 16 gamma values;
    (c) (b) at k=64, where the cluster sweep is the only pbcd sweep;  (d) one-vs-rest, 10 classes on (b)'s X,
    omegacs.
Every workload runs a fixed number of epochs (tol=-1).  Per workload: wall time of fit_many and of the loop of
single fits (after a warm-up of each), the loop both with the cluster sweep (the bit-identical reference) and
with the default "auto" sweep; model-epochs per second; launches per epoch by kernel class (sp_profile_*, in a
separate untimed run); and whether every model equals its cluster-sweep single fit bit for bit.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time
import warnings

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402
from sklearn.base import clone  # noqa: E402

import sparsepoly_b200 as S  # noqa: E402
from sparsepoly_b200 import _lib, synth  # noqa: E402

CLASSES = ["rows", "regcache", "sweep_pcd", "sweep_pbcd", "psgd_grad", "psgd_step", "prox", "plan"]


def workloads(epochs_a, epochs_bc):
    rng = np.random.RandomState(0)
    Xa = rng.randn(200, 100)
    ya = Xa[:, :5].sum(1) + 0.1 * rng.randn(200)
    grid = [S.SparseFactorizationMachineRegressor(degree=2, n_components=30, regularizer=reg, beta=b, gamma=g,
                                                   max_iter=epochs_a, tol=-1, random_state=0)
            for reg in ("l1", "squaredl12", "omegati") for g in np.logspace(-4, -0.5, 8) for b in (1e-3, 1e-2, 0.1, 1.0)]
    Xb = synth.uniform_sparse(10_000, 1_000, 50, 0)
    yb = np.where(np.asarray(Xb[:, :20].sum(1)).ravel() > np.median(np.asarray(Xb[:, :20].sum(1))), 1.0, -1.0)
    c1 = [S.SparseFactorizationMachineClassifier(degree=2, n_components=10, regularizer="squaredl12", loss="logistic",
                                                 beta=1e-3, gamma=g, max_iter=epochs_bc, tol=-1, random_state=0)
          for g in np.logspace(-5, -1, 16)]
    labels = np.random.RandomState(1).randint(0, 10, Xb.shape[0])
    ovr = [S.SparseFactorizationMachineClassifier(degree=2, n_components=10, regularizer="squaredl12", loss="logistic",
                                                  beta=1e-3, gamma=1e-3, max_iter=epochs_bc, tol=-1, random_state=0)
           for _ in range(10)]
    return [("a_notebook_grid", grid, Xa, ya), ("b_c1_shape_gamma16", c1, Xb, yb),
            ("c_one_vs_rest_10", ovr, Xb, [(labels == c).astype(float) for c in range(10)])]


def workloads_pbcd(epochs_a, epochs_bc):
    rng = np.random.RandomState(0)
    Xa = rng.randn(200, 100)
    ya = Xa[:, :5].sum(1) + 0.1 * rng.randn(200)
    grid = [S.SparseFactorizationMachineRegressor(degree=2, n_components=30, solver="pbcd", regularizer=reg, beta=b,
                                                   gamma=g, max_iter=epochs_a, tol=-1, random_state=0)
            for reg in ("l21", "squaredl21", "omegacs") for g in np.logspace(-4, -0.5, 8) for b in (1e-3, 1e-2, 0.1, 1.0)]
    Xb = synth.uniform_sparse(10_000, 1_000, 50, 0)
    yb = np.where(np.asarray(Xb[:, :20].sum(1)).ravel() > np.median(np.asarray(Xb[:, :20].sum(1))), 1.0, -1.0)

    def c1(k, reg, gamma):
        return S.SparseFactorizationMachineClassifier(degree=2, n_components=k, solver="pbcd", regularizer=reg,
                                                      loss="logistic", beta=1e-3, gamma=gamma, max_iter=epochs_bc,
                                                      tol=-1, random_state=0)
    labels = np.random.RandomState(1).randint(0, 10, Xb.shape[0])
    return [("a_notebook_grid", grid, Xa, ya),
            ("b_c1_shape_l21_gamma16", [c1(10, "l21", g) for g in np.logspace(-5, -1, 16)], Xb, yb),
            ("c_c1_shape_k64_gamma16", [c1(64, "l21", g) for g in np.logspace(-5, -1, 16)], Xb, yb),
            ("d_one_vs_rest_10", [c1(10, "omegacs", 1e-3) for _ in range(10)], Xb,
             [(labels == c).astype(float) for c in range(10)])]


def _quiet(fn):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return fn()


def _timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    r = _quiet(fn)
    torch.cuda.synchronize()
    return time.perf_counter() - t0, r


def _loop(ests, X, ys):
    return [clone(e).fit(X, yi) for e, yi in zip(ests, ys)]


def _launches(fn, epochs):
    lib = _lib.load()
    lib.sp_profile_enable(1)
    try:
        _quiet(fn)
        ms, n = (C.c_double * 8)(), (C.c_longlong * 8)()
        _lib.check(lib.sp_profile_collect(ms, n))
    finally:
        lib.sp_profile_enable(0)
    return {CLASSES[i]: n[i] / epochs for i in range(8) if n[i]}


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    return [dict(zip(q.split(","), (v.strip() for v in ln.split(",")))) for ln in out]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("outdir")
    ap.add_argument("--solver", choices=("pcd", "pbcd"), default="pcd")
    ap.add_argument("--epochs-a", type=int, default=20)
    ap.add_argument("--epochs-bc", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("fit_many_bench needs a CUDA device")
    torch.cuda.set_device(0)
    result = {"gpu": gpu_info(), "torch": torch.__version__, "workloads": {}}
    make = workloads_pbcd if args.solver == "pbcd" else workloads
    for name, ests, X, y in make(args.epochs_a, args.epochs_bc):
        ys = y if isinstance(y, list) else [y] * len(ests)
        epochs = ests[0].max_iter
        rec = {"models": len(ests), "epochs": epochs, "shape": list(X.shape)}
        os.environ["SPARSEPOLY_B200_SWEEP"] = "cluster"
        _quiet(lambda: S.fit_many([clone(e) for e in ests[:2]], X, ys[:2]))          # warm-up
        _quiet(lambda: _loop(ests[:2], X, ys[:2]))
        rec["fit_many_s"], many = _timed(lambda: S.fit_many([clone(e) for e in ests], X, ys))
        rec["loop_cluster_s"], loop = _timed(lambda: _loop(ests, X, ys))
        rec["bitwise_equal_models"] = int(sum(np.array_equal(a.P_, b.P_) and np.array_equal(a.w_, b.w_)
                                              and a.n_iter_ == b.n_iter_ for a, b in zip(many, loop)))
        rec["launches_per_epoch_fit_many"] = _launches(lambda: S.fit_many([clone(e) for e in ests], X, ys), epochs)
        rec["launches_per_epoch_loop"] = _launches(lambda: _loop(ests, X, ys), epochs)
        os.environ["SPARSEPOLY_B200_SWEEP"] = "auto"
        _quiet(lambda: _loop(ests[:2], X, ys[:2]))
        rec["loop_auto_s"], loop_auto = _timed(lambda: _loop(ests, X, ys))
        rec["auto_sweep_mode"] = "window" if (_quiet(lambda: clone(ests[0]).set_params(max_iter=1).fit(X, ys[0]))
                                              ._dev_state["plan"].mode == "window") else "cluster"
        model_epochs = len(ests) * epochs
        for key in ("fit_many_s", "loop_cluster_s", "loop_auto_s"):
            rec[key.replace("_s", "_model_epochs_per_s")] = model_epochs / rec[key]
        rec["speedup_vs_loop_cluster"] = rec["loop_cluster_s"] / rec["fit_many_s"]
        rec["speedup_vs_loop_auto"] = rec["loop_auto_s"] / rec["fit_many_s"]
        result["workloads"][name] = rec
        print(name, json.dumps(rec), flush=True)
    os.makedirs(args.outdir, exist_ok=True)
    out = "fit_many_pbcd_bench.json" if args.solver == "pbcd" else "fit_many_bench.json"
    with open(os.path.join(args.outdir, out), "w") as f:
        json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
