"""Scoring many fitted models at once against the loop of single calls; writes score_many_bench.json into OUTDIR.

    python scripts/score_many_bench.py OUTDIR [--rows-d 2000000]

Workloads: the three fit_many workloads of scripts/fit_many_bench.py (5 epochs each, pcd), scored on a held-out X
of the same shape -- (a) the notebook grid of 96 models, (b) the C1 shape with 16 gamma values, (c) one-vs-rest
with 10 classes plus the argmax over the classes -- and (d) 8 C5-shaped models (d = 1 M, k = 32, 10 % nonzero P_,
as bench.py draws its prediction model) on 2 M rows, where the per-model work is HBM-bound.
Per workload: wall time of decision_function_many and of objective_many against the loop of single calls (after a
warm-up of each, host clock around work that ends in a device synchronise); the fit_many time of the same models;
launches per call by kernel class (sp_profile_*, separate untimed runs); whether every row / objective is
bit-identical; for (d) the prediction kernel's CUDA-event time and bytes/s by the byte model of DESIGN.md 3.1; the
card's name, power limit and SM clocks, read in the same run.
"""
import argparse
import ctypes as C
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import torch  # noqa: E402

import fit_many_bench as FMB  # noqa: E402
import sparsepoly_b200 as S  # noqa: E402
from sparsepoly_b200 import _lib, synth  # noqa: E402


def gpu_info():
    import subprocess
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    return [dict(zip(q.split(","), (v.strip() for v in ln.split(",")))) for ln in out]


def _profiled(fn):
    """(result, launches by class, ms by class) of fn() with sp_profile_* on."""
    lib = _lib.load()
    lib.sp_profile_enable(1)
    try:
        r = FMB._quiet(fn)
        ms, n = (C.c_double * 8)(), (C.c_longlong * 8)()
        _lib.check(lib.sp_profile_collect(ms, n))
    finally:
        lib.sp_profile_enable(0)
    return r, {FMB.CLASSES[i]: n[i] for i in range(8) if n[i]}, {FMB.CLASSES[i]: ms[i] for i in range(8) if n[i]}


def _loop_decision(ests, X):
    return np.stack([e._predict(X) for e in ests])


def _loop_objective(ests, X, ys):
    return [S.objective(e, X, yb) for e, yb in zip(ests, ys)]


def c5_models(n_rows, n_models=8):
    X = synth.criteo_like(n_rows, 1_000_000, 0)
    d, k = X.shape[1], 32
    ests = []
    for b in range(n_models):
        rng = np.random.RandomState(b)
        e = S.SparseFactorizationMachineClassifier(degree=2, n_components=k, loss="logistic",
                                                   regularizer=("squaredl12", "l1", "omegati", "l21")[b % 4])
        e.P_ = 0.01 * rng.randn(1, k, d) * (rng.rand(1, k, d) < 0.1)        # as bench.py draws its model
        e.w_ = 0.01 * rng.randn(d)
        e.lams_ = np.ones(k)
        ests.append(e)
    y = np.where(np.random.RandomState(99).rand(n_rows) < 0.25, 1.0, -1.0)
    for e in ests:                                                           # a fitted classifier's binarizer
        e._check_X_y(X[:2], np.array([-1.0, 1.0]))
    return ests, X, y


def measure(name, ests, X, ys, fit_s, argmax=False):
    rec = {"models": len(ests), "shape": list(X.shape), "fit_many_s": fit_s}
    FMB._quiet(lambda: S.decision_function_many(ests[:2], X))                # warm-up of every shape used
    FMB._quiet(lambda: _loop_decision(ests[:2], X))
    FMB._quiet(lambda: S.objective_many(ests[:2], X, ys[:2]))
    FMB._quiet(lambda: _loop_objective(ests[:2], X, ys[:2]))

    def many_dec():
        dec = S.decision_function_many(ests, X)
        return (dec, dec.argmax(axis=0)) if argmax else (dec, None)

    def loop_dec():
        dec = _loop_decision(ests, X)
        return (dec, dec.argmax(axis=0)) if argmax else (dec, None)
    rec["decision_many_s"], (dm, am) = FMB._timed(many_dec)
    rec["decision_loop_s"], (dl, al) = FMB._timed(loop_dec)
    rec["objective_many_s"], om = FMB._timed(lambda: S.objective_many(ests, X, ys))
    rec["objective_loop_s"], ol = FMB._timed(lambda: _loop_objective(ests, X, ys))
    rec["decision_speedup"] = rec["decision_loop_s"] / rec["decision_many_s"]
    rec["objective_speedup"] = rec["objective_loop_s"] / rec["objective_many_s"]
    if fit_s:
        rec["scoring_share_of_fit_plus_score_many"] = (rec["decision_many_s"] + rec["objective_many_s"]) / (
            fit_s + rec["decision_many_s"] + rec["objective_many_s"])
        rec["scoring_share_of_fit_plus_score_loop"] = (rec["decision_loop_s"] + rec["objective_loop_s"]) / (
            fit_s + rec["decision_loop_s"] + rec["objective_loop_s"])
    rec["bitwise_equal_rows"] = int(sum(np.array_equal(a, b) for a, b in zip(dm, dl)))
    rec["bitwise_equal_objectives"] = int(sum(a == b for a, b in zip(om, ol)))
    if argmax:
        rec["argmax_equal"] = bool(np.array_equal(am, al))
    _, rec["launches_decision_many"], ms = _profiled(lambda: S.decision_function_many(ests, X))
    _, rec["launches_decision_loop"], _ = _profiled(lambda: _loop_decision(ests, X))
    _, rec["launches_objective_many"], _ = _profiled(lambda: S.objective_many(ests, X, ys))
    _, rec["launches_objective_loop"], _ = _profiled(lambda: _loop_objective(ests, X, ys))
    rec["rows_kernel_ms_decision_many"] = ms.get("rows")
    print(name, json.dumps(rec), flush=True)
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("outdir")
    ap.add_argument("--rows-d", type=int, default=2_000_000)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("score_many_bench needs a CUDA device")
    torch.cuda.set_device(0)
    result = {"gpu": gpu_info(), "torch": torch.__version__, "workloads": {}}
    os.environ["SPARSEPOLY_B200_SWEEP"] = "cluster"
    held_out = {"a_notebook_grid": np.random.RandomState(5).randn(200, 100),
                "b_c1_shape_gamma16": synth.uniform_sparse(10_000, 1_000, 50, 5)}
    held_out["c_one_vs_rest_10"] = held_out["b_c1_shape_gamma16"]
    for name, ests, X, y in FMB.workloads(5, 5):
        ys = y if isinstance(y, list) else [y] * len(ests)
        FMB._quiet(lambda: S.fit_many([e for e in ests[:2]], X, ys[:2]))   # warm-up
        fit_s, _ = FMB._timed(lambda: S.fit_many(ests, X, ys))
        Xh = held_out[name]
        rng = np.random.RandomState(6)
        if name.startswith("a"):
            yh = [Xh[:, :5].sum(1) + 0.1 * rng.randn(Xh.shape[0])] * len(ests)
        elif name.startswith("b"):
            s = np.asarray(Xh[:, :20].sum(1)).ravel()
            yh = [np.where(s > np.median(s), 1.0, -1.0)] * len(ests)
        else:
            labels = rng.randint(0, 10, Xh.shape[0])
            yh = [(labels == c).astype(float) for c in range(10)]
        result["workloads"][name] = measure(name, ests, Xh, yh, fit_s, argmax=name.startswith("c"))
    ests, X, y = c5_models(args.rows_d)
    rec = measure("d_c5_8_models", ests, X, [y] * len(ests), None)
    r = X.nnz / X.shape[0]
    k = ests[0].n_components
    per_sample = r * 12 + r * k * 8 + r * 8 + 8                 # DESIGN.md 3.1, one output order
    ms = rec["rows_kernel_ms_decision_many"]
    rec["predict_bytes_model"] = per_sample * X.shape[0] * len(ests)
    rec["predict_bytes_per_s"] = rec["predict_bytes_model"] / (ms / 1e3) if ms else None
    result["workloads"]["d_c5_8_models"] = rec
    result["gpu_after"] = gpu_info()
    os.makedirs(args.outdir, exist_ok=True)
    with open(os.path.join(args.outdir, "score_many_bench.json"), "w") as f:
        json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
