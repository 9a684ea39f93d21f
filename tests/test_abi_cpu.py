"""CPU-side checks of the drop-in boundary: the shared library loads, exports every symbol the
header declares, and the host logic (validation, sharding helpers) behaves.  No compute calls."""
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header_symbols():
    src = open(os.path.join(ROOT, "include", "sparsepoly_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(sp_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    from sparsepoly_b200 import _lib
    lib = _lib.load()
    declared = _header_symbols()
    assert len(declared) >= 18
    for name in declared:
        assert hasattr(lib, name), name
        assert name in _lib.SIGNATURES, f"{name} has no ctypes signature"
    assert set(_lib.SIGNATURES) == set(declared)
    assert lib.sp_abi_version() == 4


def test_get_eta_matches_oracle():
    # psgd.py:9-22 (host scalar helper of the ABI; no GPU needed)
    import ctypes as C
    from oracle import oracle as O
    from sparsepoly_b200 import solvers
    for lr in range(4):
        for it in (1, 7, 1000):
            a, b = C.c_double(), C.c_double()
            O.lib().sp_oracle_get_eta(lr, 0.3, 0.2, 0.7, 0.8, it, C.byref(a), C.byref(b))
            assert solvers.get_eta(lr, 0.3, 0.2, 0.7, 0.8, it) == (a.value, b.value)


def test_rec_stride():
    from sparsepoly_b200 import solvers
    assert [solvers.rec_stride(m) for m in (-1, 2, 3, 4, 5)] == [4, 4, 4, 8, 8]


def test_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    import sparsepoly_b200 as S
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        S.SparseFactorizationMachineRegressor().fit(np.random.randn(10, 3), np.random.randn(10))


def test_validation_errors_before_device_work():
    import sparsepoly_b200 as S
    X, y = np.random.randn(12, 3), np.random.randn(12)
    with pytest.raises(ValueError, match="Regularizer foo not supported"):
        S.SparseFactorizationMachineRegressor(regularizer="foo").fit(X, y)
    with pytest.raises(ValueError, match="Solver sgd is not supported"):
        S.SparseFactorizationMachineRegressor(solver="sgd").fit(X, y)
    with pytest.raises(ValueError, match="cannot be used with solver pcd"):
        S.SparseFactorizationMachineRegressor(solver="pcd", regularizer="l21").fit(X, y)
    with pytest.raises(ValueError, match="SquaredL12 supports only degree=2"):
        S.SparseFactorizationMachineRegressor(degree=3, regularizer="squaredl12").fit(X, y)
    with pytest.raises(ValueError, match="SquaredL21 supports only degree=2"):
        S.SparseFactorizationMachineRegressor(degree=3, solver="pbcd", regularizer="squaredl21").fit(X, y)
    with pytest.raises(ValueError, match="Loss function hinge not supported"):
        S.SparseFactorizationMachineClassifier(loss="hinge").fit(X, np.sign(y))
    with pytest.raises(TypeError, match="Only binary targets supported"):
        S.SparseFactorizationMachineClassifier().fit(X, np.arange(12) % 3)
    with pytest.raises(ValueError, match="not supported"):
        S.SparseAllSubsetsRegressor(regularizer="squaredl12").fit(X, y)


def test_public_surface_matches_reference_signatures():
    import inspect
    import sparsepoly_b200 as S
    fm = inspect.signature(S.SparseFactorizationMachineClassifier.__init__).parameters
    assert list(fm)[1:] == ["degree", "loss", "n_components", "solver", "regularizer", "alpha", "beta",
                            "gamma", "mean", "tol", "fit_lower", "fit_linear", "warm_start",
                            "init_lambdas", "max_iter", "shuffle", "batch_size", "eta0",
                            "learning_rate", "power_t", "n_iter_no_change", "verbose", "callback",
                            "n_calls", "random_state"]
    assert fm["loss"].default == "squared_hinge" and fm["regularizer"].default == "squaredl12"
    al = inspect.signature(S.SparseAllSubsetsRegressor.__init__).parameters
    assert list(al)[1:] == ["n_components", "solver", "beta", "gamma", "eta0", "mean", "tol",
                            "regularizer", "warm_start", "init_lambdas", "max_iter", "shuffle",
                            "verbose", "callback", "n_calls", "random_state"]
    assert al["eta0"].default == 0.1 and al["regularizer"].default == "omegati"
    est = S.SparseFactorizationMachineRegressor(degree=3, gamma=0.5)
    assert est.get_params()["degree"] == 3 and est.set_params(gamma=2).gamma == 2


def test_local_batches_cover_reference_minibatches():
    from sparsepoly_b200.distributed import interleave_shards, local_batches
    n_local, world, B = 23, 2, 8
    bs = list(local_batches(n_local, B, world))
    assert bs[0] == (0, 4, 8) and bs[-1] == (20, 23, 6)
    assert sum(b1 - b0 for b0, b1, _ in bs) == n_local
    shards = [np.arange(0, 23), np.arange(100, 123)]
    order = interleave_shards(shards, B)
    assert order[:8].tolist() == [0, 1, 2, 3, 100, 101, 102, 103]
    assert sorted(order.tolist()) == sorted(np.concatenate(shards).tolist())


def test_ctypes_structs_match_the_header_layout(tmp_path):
    """sizeof / offsetof of every struct of include/sparsepoly_b200.h (compiled with gcc) against the
    ctypes mirrors in sparsepoly_b200/_lib.py: a renamed or reordered field must not go unnoticed."""
    import ctypes as C
    import shutil
    import subprocess
    from sparsepoly_b200 import _lib
    if shutil.which("gcc") is None:
        pytest.skip("gcc not available")
    mirrors = {"sp_dataset": _lib.SpDataset, "sp_plan": _lib.SpPlan, "sp_wplan": _lib.SpWPlan,
               "sp_psgd_plan": _lib.SpPsgdPlan, "sp_psgd_ctx": _lib.SpPsgdCtx}
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "sparsepoly_b200.h"', "int main(void) {"]
    for cname, cls in mirrors.items():
        lines.append(f'  printf("{cname} size %zu\\n", sizeof(struct {cname}));')
        for fname, _ in cls._fields_:
            lines.append(f'  printf("{cname} {fname} %zu\\n", offsetof(struct {cname}, {fname}));')
    lines += ["  return 0;", "}"]
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)])
    got = {}
    for ln in subprocess.check_output([str(exe)], text=True).splitlines():
        cname, field, val = ln.split()
        got[(cname, field)] = int(val)
    for cname, cls in mirrors.items():
        assert got[(cname, "size")] == C.sizeof(cls), cname
        for fname, _ in cls._fields_:
            assert got[(cname, fname)] == getattr(cls, fname).offset, (cname, fname)


def test_fitted_estimators_pickle_without_device_state():
    """ADVICE r1: _dev_state holds ctypes structs with pointers; a fitted estimator must still pickle."""
    import ctypes as C
    import copy
    import pickle
    import sparsepoly_b200 as S
    from sparsepoly_b200 import _lib
    est = S.SparseFactorizationMachineRegressor(degree=2, n_components=3)
    est.P_ = np.zeros((1, 3, 5)); est.w_ = np.zeros(5); est.lams_ = np.ones(3); est.n_iter_ = 4
    est._dev_state = {"ds": _lib.SpDataset(), "plan": C.pointer(_lib.SpPlan())}      # what fit leaves behind
    est2 = pickle.loads(pickle.dumps(est))
    assert np.array_equal(est2.P_, est.P_) and est2.n_iter_ == 4 and not hasattr(est2, "_dev_state")
    est3 = copy.deepcopy(est)
    assert not hasattr(est3, "_dev_state") and est3.get_params() == est.get_params()


def test_binary_label_fast_path_equals_label_binarizer():
    """Classifier._binary_labels (a few streaming passes) must give what the reference's
    type_of_target + LabelBinarizer(pos_label=1, neg_label=-1) give (base.py:126-142), and must step aside
    for everything else."""
    from sklearn.preprocessing import LabelBinarizer

    from sparsepoly_b200.estimators import SparsePolyClassifierMixin as Mixin
    rng = np.random.RandomState(0)
    for y in (rng.randint(0, 2, 64), np.where(rng.rand(64) < 0.3, 1.0, -1.0), rng.randint(0, 2, 64) * 3 + 2,
              rng.randint(0, 2, 64).astype(np.uint8), rng.randint(0, 2, 64).astype(np.float32)):
        fast = Mixin._binary_labels(y)
        lb = LabelBinarizer(pos_label=1, neg_label=-1)
        want = lb.fit_transform(y).ravel().astype(np.double)
        assert fast is not None and np.array_equal(fast[1], want) and np.array_equal(fast[0], lb.classes_)
        lb2 = LabelBinarizer(pos_label=1, neg_label=-1)
        lb2.classes_, lb2.y_type_, lb2.sparse_input_ = fast[0], "binary", False
        yp = rng.rand(64) > 0.5
        assert np.array_equal(lb2.inverse_transform(yp), lb.inverse_transform(yp))
        assert lb2.inverse_transform(yp).dtype == lb.inverse_transform(yp).dtype
    for y in (rng.rand(16), rng.randint(0, 3, 64), np.array([1.0, 1.0]), np.array([0.5, 1.5, 0.5]),
              np.array(["a", "b"]), np.array([0.0, np.nan, 1.0]), np.array([0.0, np.inf]), np.zeros((4, 1)),
              [0, 1, 0], np.array([True, False])):
        assert Mixin._binary_labels(y) is None


def test_upload_thread_errors_reach_the_caller():
    """fit() moves X to the device on a helper thread (estimators._start_upload); whatever goes wrong there must be
    raised by the joining thread, not swallowed.  Without a GPU the helper fails at once: exactly that case."""
    import scipy.sparse as sp
    import torch

    import sparsepoly_b200 as S
    if torch.cuda.is_available():
        pytest.skip("needs a box without CUDA")
    est = S.SparseFactorizationMachineClassifier(solver="psgd", regularizer="squaredl12", n_components=2)
    X = sp.random(20, 5, density=0.5, format="csr", random_state=0)
    y = np.where(np.arange(20) % 2 == 0, 1.0, -1.0)
    dev = torch.device("cuda", 0)
    upload = est._start_upload(X, dev)
    upload[0].join()
    assert "error" in upload[1] and "ds" not in upload[1]
    est.P_, est.w_, est.lams_, est.it_ = np.zeros((1, 2, 5)), np.zeros(5), np.ones(2), 1
    with pytest.raises(type(upload[1]["error"])):
        est._psgd_setup(X, y, np.random.RandomState(0), dev, upload)
