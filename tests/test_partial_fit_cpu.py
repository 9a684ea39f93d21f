"""partial_fit input errors: each is a clean ValueError raised before any device work (on a box without CUDA the
first device call would raise RuntimeError, so a ValueError here shows nothing reached the device)."""
import os
import sys

import numpy as np
import pytest
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _clf(**kw):
    import sparsepoly_b200 as S
    return S.SparseFactorizationMachineClassifier(solver="psgd", regularizer="squaredl12", **kw)


def test_partial_fit_errors_before_device_work():
    import sparsepoly_b200 as S
    X, y = np.random.RandomState(0).randn(12, 3), np.where(np.arange(12) % 2 == 0, 1.0, -1.0)
    for solver in ("pcd", "pbcd"):
        with pytest.raises(ValueError, match="psgd"):
            S.SparseFactorizationMachineRegressor(solver=solver).partial_fit(X, y)
    with pytest.raises(ValueError, match="cannot be used with solver psgd"):
        S.SparseFactorizationMachineRegressor(solver="psgd", regularizer="omegati").partial_fit(X, y)
    with pytest.raises(ValueError, match="learning_rate"):
        S.SparseFactorizationMachineRegressor(solver="psgd", learning_rate="adaptive").partial_fit(X, y)
    # classes: required on the first call, exactly two labels
    with pytest.raises(ValueError, match="classes must be passed"):
        _clf().partial_fit(X, y)
    for classes in ([1.0], [-1.0, 0.0, 1.0], [1.0, 1.0], [[-1.0, 1.0]]):
        with pytest.raises(ValueError, match="exactly two"):
            _clf().partial_fit(X, y, classes=classes)
    with pytest.raises(ValueError, match="not in classes"):
        _clf().partial_fit(X, np.where(y > 0, 2.0, -1.0), classes=[-1.0, 1.0])
    est = _clf()
    with pytest.raises(ValueError, match="not in classes"):
        est.partial_fit(X, np.array(["a", "b", "c"] * 4), classes=["a", "b"])
    assert not hasattr(est, "label_binarizer_")          # a refused first call leaves no state behind
    # n_features of the stream (after the augment columns)
    est = S.SparseFactorizationMachineRegressor(solver="psgd", regularizer="l1", degree=3, fit_lower="augment",
                                                fit_linear=True)
    est.P_, est.w_, est.lams_, est.it_ = np.zeros((1, 2, 4)), np.zeros(4), np.ones(2), 1
    with pytest.raises(ValueError, match="X has 5 features"):
        est.partial_fit(np.random.randn(12, 4), np.random.randn(12))
    # a model of another shape (set_params after fit / mid-stream)
    est.set_params(n_components=3)
    with pytest.raises(ValueError, match="shape"):
        est.partial_fit(np.random.randn(12, 3), np.random.randn(12))


def test_partial_fit_refuses_changes_mid_stream():
    from sklearn.preprocessing import LabelBinarizer
    X, y = np.random.RandomState(0).randn(12, 3), np.where(np.arange(12) % 2 == 0, 1.0, -1.0)
    est = _clf(n_components=2)
    est.P_, est.w_, est.lams_, est.it_ = np.zeros((1, 2, 3)), np.zeros(3), np.ones(2), 1
    est.label_binarizer_ = LabelBinarizer(pos_label=1, neg_label=-1).fit([-1.0, 1.0])
    with pytest.raises(ValueError, match="differs from the classes"):
        est.partial_fit(X, y, classes=[0.0, 1.0])
    est._psgd_stream = {"config": est._stream_config(), "ctx": None}      # what a first call leaves behind
    est.set_params(regularizer="l1")
    with pytest.raises(ValueError, match="changed since the stream started"):
        est.partial_fit(X, y)


def test_partial_fit_without_a_device_fails_loudly():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        _clf().partial_fit(np.random.randn(10, 3), np.where(np.arange(10) % 2 == 0, 1.0, -1.0), classes=[-1.0, 1.0])


def _sharded_worker(rank, world, port):
    sys.path.insert(0, ROOT)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from sparsepoly_b200 import distributed
    est = _clf()
    X, y = np.random.randn(10, 3), np.where(np.arange(10) % 2 == 0, 1.0, -1.0)
    with distributed.sharded():
        try:
            est.partial_fit(X, y, classes=[-1.0, 1.0])
            raise AssertionError("sharded partial_fit accepted")
        except ValueError as e:
            assert "enable_sharding" in str(e), e
    dist.destroy_process_group()


def test_partial_fit_refuses_sharding():
    world = 2
    port = 33500 + (os.getpid() % 2000)
    mp.spawn(_sharded_worker, args=(world, port), nprocs=world, join=True)
