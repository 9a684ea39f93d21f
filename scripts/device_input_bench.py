"""Host X against CUDA X on the same rows; writes device_input_bench.json into OUTDIR.

    python scripts/device_input_bench.py OUTDIR [--rows 6250000] [--d 1000000] [--chunk 1250000] [--reps 2]

(a) the C5 psgd fit of bench.py (Criteo-shaped X: 13 dense + 26 Zipf one-hot fields, d = 1M; planted degree-2
    targets; k = 32, squaredl12, logistic, batch_size "auto"), one epoch: wall time of fit() and its
    _psgd_stats["setup_seconds"] (SPARSEPOLY_B200_TIMING=1: the phases end in a device synchronise), and the time of
    the input check alone (_check_X_y);
(b) the partial_fit stream of DESIGN.md 7 (chunks of ~1.23 M rows, 2 passes): the per-call phases of
    _partial_fit_stats, summed over the calls;
(c) decision_function on 2 M C5 rows;
(d) sp_csr_prepare alone on the C5 matrix, CUDA events over repeated launches: check only (canonical int32 / fp64, the
    zero-copy case), and check + conversion from int32 / fp64 and from int64 indices / fp32 values; GB/s from the bytes
    the kernel must read and write (computed from the shapes).
The CUDA X is uploaded before any timed region.  Every host / device pair must give bit-identical models and outputs;
the JSON says whether they did.  Host and device runs alternate, after a warm-up of both paths at a small size.
"""
import argparse
import json
import os
import subprocess
import sys
import time
import warnings

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
os.environ["SPARSEPOLY_B200_TIMING"] = "1"

import torch  # noqa: E402

import sparsepoly_b200 as S  # noqa: E402
from sparsepoly_b200 import dataset, synth  # noqa: E402

KW = dict(degree=2, loss="logistic", n_components=32, solver="psgd", regularizer="squaredl12", alpha=1e-7, beta=1e-7,
          gamma=2e-8, fit_linear=True, fit_lower="explicit", batch_size="auto", eta0=0.1, learning_rate="optimal",
          power_t=1.0, shuffle=False, random_state=0, tol=-1.0, n_iter_no_change=10 ** 9)
FMC = S.SparseFactorizationMachineClassifier


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i",
                          str(torch.cuda.current_device())], capture_output=True, text=True, timeout=60).stdout.strip()
    name, plim, sm, smax = [c.strip() for c in out.split(",")]
    return {"name": name, "power_limit": plim, "sm_clock": sm, "sm_clock_max": smax}


def cuda_csr(X, index=torch.int32, value=torch.float64):
    t = lambda a, dt: torch.from_numpy(a).to(dt)                    # noqa: E731
    return torch.sparse_csr_tensor(t(X.indptr, index), t(X.indices, index), t(X.data, value), size=X.shape,
                                   device="cuda")


def clock(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, out


def fit_once(X, y, max_iter):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return clock(lambda: FMC(max_iter=max_iter, **KW).fit(X, y))


def same_model(a, b):
    return bool(np.array_equal(a.P_, b.P_) and np.array_equal(a.w_, b.w_) and a.it_ == b.it_)


def part_a(X, Xd, y, reps):
    res = {"host": [], "device": []}
    models = {}
    for _ in range(reps):
        for tag, Xi in (("host", X), ("device", Xd)):
            t_check, _ = clock(lambda: FMC(**KW)._check_X_y(Xi, y))
            t_fit, est = fit_once(Xi, y, 1)
            res[tag].append({"fit_s": t_fit, "check_X_y_s": t_check, "setup_seconds": est._psgd_stats["setup_seconds"]})
            models[tag] = est
    res["bit_identical"] = same_model(models["host"], models["device"])
    res["samples_per_s"] = {t: X.shape[0] / min(r["fit_s"] for r in res[t]) for t in ("host", "device")}
    return res, models["host"]


def part_b(X, y, chunk, passes):
    chunks = [(X[a:a + chunk], y[a:a + chunk]) for a in range(0, X.shape[0], chunk)]
    dev_chunks = [(cuda_csr(Xc), yc) for Xc, yc in chunks]           # uploaded before the timed region
    torch.cuda.synchronize()
    out, models = {}, {}
    for tag, cs in (("host", chunks), ("device", dev_chunks)):
        est = FMC(**KW)
        calls = []
        for _ in range(passes):
            for Xc, yc in cs:
                t, _ = clock(lambda: est.partial_fit(Xc, yc, classes=[-1.0, 1.0]))
                calls.append(dict(est._partial_fit_stats, call_s=t))
        phases = ["validate_s", "h2d_s", "model_s", "plan_s", "minibatches_s", "readout_s", "call_s"]
        steady = calls[1:]                                            # (the first call also draws the model)
        out[tag] = {"calls": calls, "phase_totals_s": {p: float(sum(c[p] for c in calls)) for p in phases},
                    "steady_call_mean_s": {p: float(np.mean([c[p] for c in steady])) for p in phases}}
        models[tag] = est
    out["chunk_rows"], out["calls"] = chunk, len(chunks) * passes
    out["bit_identical"] = same_model(models["host"], models["device"])
    return out


def part_c(est, X, reps):
    Xd = cuda_csr(X)
    torch.cuda.synchronize()
    res = {"host": [], "device": []}
    outs = {}
    for _ in range(reps):
        for tag, Xi in (("host", X), ("device", Xd)):
            t, outs[tag] = clock(lambda: est.decision_function(Xi))
            res[tag].append(t)
    res["rows"] = X.shape[0]
    res["bit_identical"] = bool(np.array_equal(outs["host"], outs["device"]))
    return res


def part_d(X, launches):
    n, d, nnz = X.shape[0], X.shape[1], X.nnz
    dev = torch.device("cuda")
    src32 = [torch.from_numpy(a).to(dev) for a in (X.indptr.astype(np.int32), X.indices, X.data)]
    src64 = [torch.from_numpy(X.indptr.astype(np.int64)).to(dev), torch.from_numpy(X.indices.astype(np.int64)).to(dev),
             torch.from_numpy(X.data.astype(np.float32)).to(dev)]
    out = dataset._alloc_csr(n, nnz, dev)
    cases = {
        "check_only_int32_fp64": (src32, None, (n + 1) * 4 + nnz * 12, X),
        "convert_int32_fp64": (src32, out, (n + 1) * 4 + nnz * 12 + (n + 1) * 4 + nnz * 12, X),
        "convert_int64_fp32": (src64, out, (n + 1) * 8 + nnz * 12 + (n + 1) * 4 + nnz * 12, X.astype(np.float32)),
    }
    res = {"rows": n, "cols": d, "nnz": nnz, "launches": launches}
    for name, (src, o, nbytes, X_same) in cases.items():
        report = None
        for _ in range(3):                                            # warm-up
            report = dataset._run_prepare(n, d, *src, (0, 0), 0, o)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(launches):
            dataset._run_prepare(n, d, *src, (0, 0), 0, o)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / launches
        res[name] = {"ms_per_launch": ms, "bytes": nbytes, "GB_per_s": nbytes / (ms * 1e-3) / 1e9,
                     "report_clean": report.tolist()[3:] == [2 ** 63 - 1] * 3 + [0, 2 ** 63 - 1]}
        if o is not None:
            want = dataset.host_csr(X_same)                         # (the host path given the same fp32 matrix)
            res[name]["output_equals_host_csr"] = all(np.array_equal(t.cpu().numpy(), w) for t, w in zip(o, want))
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("outdir")
    ap.add_argument("--rows", type=int, default=6_250_000)
    ap.add_argument("--d", type=int, default=1_000_000)
    ap.add_argument("--chunk", type=int, default=1_250_000)
    ap.add_argument("--passes", type=int, default=2)
    ap.add_argument("--predict-rows", type=int, default=2_000_000)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--launches", type=int, default=20)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "the benchmark needs a CUDA device"
    os.makedirs(args.outdir, exist_ok=True)
    info = gpu_info()
    t0 = time.perf_counter()
    X = synth.criteo_like(args.rows, args.d, 4000)
    y = synth.planted_fm_targets(X, 4, 99, positive_frac=0.25)
    t_gen = time.perf_counter() - t0
    batch = int(X.shape[0] * X.shape[1] / X.nnz)
    chunk = max(args.chunk // batch, 1) * batch
    n_stream = max(args.rows // chunk, 1) * chunk
    # warm-up of every path at a small size (module loads, allocator)
    w = 4 * chunk // 64
    fit_once(X[:w], y[:w], 1)
    fit_once(cuda_csr(X[:w]), y[:w], 1)
    part_b(X[:4 * batch], y[:4 * batch], batch, 1)
    Xd = cuda_csr(X)
    torch.cuda.synchronize()
    a, est = part_a(X, Xd, y, args.reps)
    del Xd
    b = part_b(X[:n_stream], y[:n_stream], chunk, args.passes)
    c = part_c(est, X[:args.predict_rows], args.reps)
    d = part_d(X, args.launches)
    result = {"gpu": info, "workload": {"rows": X.shape[0], "d": args.d, "nnz": int(X.nnz), "batch_size": batch,
                                        "estimator": KW, "data_generation_s": t_gen},
              "a_psgd_fit": a, "b_partial_fit": b, "c_decision_function": c, "d_sp_csr_prepare": d,
              "gpu_after": gpu_info()}
    with open(os.path.join(args.outdir, "device_input_bench.json"), "w") as f:
        json.dump(result, f, indent=1)
    summary = {"gpu": info, "a": {k: a[k] for k in ("samples_per_s", "bit_identical")},
               "b": {t: b[t]["steady_call_mean_s"] for t in ("host", "device")}, "b_same": b["bit_identical"],
               "c": c, "d": {k: v for k, v in d.items() if isinstance(v, dict)}}
    print(json.dumps(summary))


if __name__ == "__main__":
    main()
