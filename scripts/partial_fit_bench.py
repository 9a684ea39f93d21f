"""Streaming psgd: partial_fit over C5-shaped chunks against fit on the same rows; writes partial_fit_bench.json into
OUTDIR.

    python scripts/partial_fit_bench.py OUTDIR [--rows 6250000] [--chunk 1250000] [--d 1000000] [--passes 2]

The C5 workload of bench.py (Criteo-shaped X: 13 dense + 26 Zipf one-hot fields, d = 1M; planted degree-2 targets,
25 % positives; k = 32, squaredl12, logistic, batch_size "auto") is cut into chunks of --chunk rows (a multiple of
the resolved batch size, so the stream computes what fit computes).  Per partial_fit call the estimator's own phase
split is recorded: input validation (host clock), H2D of the chunk, the model's draw + upload (first call only), plan
build and the minibatches (CUDA events),
read-out of P_ / w_ + D2H (host clock around the synchronising copy).  The same rows go through fit(max_iter=passes)
end to end (upload, plan, epochs, D2H), timed by the host clock.  After a warm-up of both paths at a small size.
Both results must be equal bit for bit; the JSON says whether they were.
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

import torch  # noqa: E402

import sparsepoly_b200 as S  # noqa: E402
from sparsepoly_b200 import synth  # noqa: E402

KW = dict(degree=2, loss="logistic", n_components=32, solver="psgd", regularizer="squaredl12", alpha=1e-7, beta=1e-7,
          gamma=2e-8, fit_linear=True, fit_lower="explicit", eta0=0.1, learning_rate="optimal", power_t=1.0,
          shuffle=False, random_state=0, tol=-1.0, n_iter_no_change=10 ** 9)


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, plim, sm, smax = [c.strip() for c in out.split(",")]
        return {"name": name, "power_limit": plim, "sm_clock": sm, "sm_clock_max": smax}
    except Exception as e:          # the torch name is still known
        return {"name": torch.cuda.get_device_name(0), "nvidia_smi": repr(e)}


def run(X, y, chunk, passes, batch_size):
    kw = dict(KW, batch_size=batch_size)
    n = X.shape[0]
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        full = S.SparseFactorizationMachineClassifier(max_iter=passes, **kw).fit(X, y)
        torch.cuda.synchronize()
        t_fit = time.perf_counter() - t0
    est = S.SparseFactorizationMachineClassifier(**kw)
    chunks = [(X[a:a + chunk], y[a:a + chunk]) for a in range(0, n, chunk)]      # (host slicing is not timed)
    calls = []
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(passes):
        for Xc, yc in chunks:
            c0 = time.perf_counter()
            est.partial_fit(Xc, yc, classes=[-1.0, 1.0])
            calls.append(dict(est._partial_fit_stats, call_s=time.perf_counter() - c0))
    t_stream = time.perf_counter() - t0
    same = bool(np.array_equal(est.P_, full.P_) and np.array_equal(est.w_, full.w_) and est.it_ == full.it_)
    return t_fit, t_stream, calls, same


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("outdir")
    ap.add_argument("--rows", type=int, default=6_250_000)
    ap.add_argument("--chunk", type=int, default=1_250_000)
    ap.add_argument("--d", type=int, default=1_000_000)
    ap.add_argument("--passes", type=int, default=2)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "the benchmark needs a CUDA device"
    os.makedirs(args.outdir, exist_ok=True)
    t0 = time.perf_counter()
    X = synth.criteo_like(args.rows, args.d, 4000)
    y = synth.planted_fm_targets(X, 4, 99, positive_frac=0.25)
    t_gen = time.perf_counter() - t0
    batch = int(X.shape[0] * X.shape[1] / X.nnz)                  # what "auto" resolves to (39 nonzeros per row)
    chunk = max(args.chunk // batch, 1) * batch
    n = max(args.rows // chunk, 1) * chunk                          # whole chunks: the stream computes what fit computes
    X, y = X[:n], y[:n]
    # warm-up of both paths (module loads, allocator) at a small size
    w = max(chunk // 16, batch)
    run(X[:4 * w], y[:4 * w], w, 1, batch)
    t_fit, t_stream, calls, same = run(X, y, chunk, args.passes, batch)
    rows = n * args.passes
    phases = ["validate_s", "h2d_s", "model_s", "plan_s", "minibatches_s", "readout_s", "call_s"]
    tot = {p: float(sum(c[p] for c in calls)) for p in phases}
    result = {
        "gpu": gpu_info(),
        "workload": {"rows": n, "d": args.d, "nnz_per_row": 39, "passes": args.passes, "chunk_rows": chunk,
                     "calls": len(calls), "batch_size": batch, "estimator": KW, "data_generation_s": t_gen},
        "fit": {"seconds": t_fit, "samples_per_s": rows / t_fit},
        "partial_fit": {"seconds": t_stream, "samples_per_s": rows / t_stream, "phase_totals_s": tot,
                        "phase_share": {p: tot[p] / tot["call_s"] for p in phases[:-1]},
                        "minibatch_samples_per_s": rows / tot["minibatches_s"]},
        "bit_identical_to_fit": same,
        "calls": calls,
    }
    with open(os.path.join(args.outdir, "partial_fit_bench.json"), "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps({k: result[k] for k in ("gpu", "fit", "partial_fit", "bit_identical_to_fit")}))


if __name__ == "__main__":
    main()
