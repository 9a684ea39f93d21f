"""Loads tests/golden/reference_fits.* (outputs of the unmodified reference, produced by
oracle/gen_golden.py)."""
import json
import os

import numpy as np
import scipy.sparse as sp

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

with open(os.path.join(GOLD, "reference_fits.json")) as _f:
    INDEX = json.load(_f)
_BLOB = None


def blob():
    global _BLOB
    if _BLOB is None:
        _BLOB = np.load(os.path.join(GOLD, "reference_fits.npz"))
    return _BLOB


def case_names(prefix=""):
    return [c["name"] for c in INDEX if c["name"].startswith(prefix)]


def load_case(name):
    rec = next(c for c in INDEX if c["name"] == name)
    b = blob()
    arr = {k.split("/", 1)[1]: b[k] for k in b.files if k.startswith(name + "/")}
    if "X_dense" in arr:
        X = arr["X_dense"]
    else:
        X = sp.csr_matrix((arr["X_data"], arr["X_indices"], arr["X_indptr"]),
                          shape=tuple(arr["X_shape"]))
    return rec, X, arr


def rel_err(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    den = max(np.max(np.abs(b)), 1e-300)
    return float(np.max(np.abs(a - b)) / den)


def same_support(a, b, noise=1e-12):
    """Identical support sets, ignoring entries that are numerical dust in BOTH arrays
    (|.| < noise * max|b|): OmegaTI/OmegaCS shrink coordinates geometrically towards 0 without
    ever thresholding them, leaving 1e-30..1e-100 residues whose sign/zero-ness is rounding
    noise even between two runs of the reference on different libm builds."""
    a = np.asarray(a)
    b = np.asarray(b)
    floor = noise * max(np.max(np.abs(b)), 1e-300)
    dust = (np.abs(a) < floor) & (np.abs(b) < floor)
    return bool(np.all(((a != 0) == (b != 0)) | dust))


# ------------------------------------------------------------------ larger reference fits (oracle/gen_golden_large.py)
with open(os.path.join(GOLD, "reference_large.json")) as _f:
    LARGE_INDEX = json.load(_f)


def large_case_names():
    return [c["name"] for c in LARGE_INDEX]


def large_inputs(prob):
    """X of a reference_large case, regenerated from the seeded generators (same code as the generating script)."""
    from sparsepoly_b200 import synth
    if prob["gen"] == "uniform":
        return synth.uniform_sparse(prob["n"], prob["d"], prob["r"], prob["seed"])
    return synth.criteo_like(prob["n"], prob["d"], prob["seed"])


def load_large_case(name):
    rec = next(c for c in LARGE_INDEX if c["name"] == name)
    with np.load(os.path.join(GOLD, "reference_large", name + ".npz")) as z:
        arr = {k: z[k] for k in z.files}
    X = large_inputs(rec["prob"])
    nnz, dsum, isum = rec["x_checksum"]
    assert X.nnz == nnz and float(X.data.sum()) == dsum and int(X.indices.astype(np.int64).sum()) == isum, \
        "regenerated inputs differ from the ones the reference was run on"
    arr["y"] = arr["y"].astype(np.float64)
    arr["Xte"] = large_inputs(dict(rec["prob"], n=200, seed=rec["prob"]["seed"] + 7))
    return rec, X, arr
