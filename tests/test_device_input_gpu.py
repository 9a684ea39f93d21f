"""X as a CUDA tensor (dataset.check_X, csrc/input.cu): every entry point must give exactly what the host path gives
for the same matrix -- fitted attributes, predictions, objectives and scores bit for bit -- and the check kernel's
report must match a numpy restatement."""
import os
import warnings

import numpy as np
import pytest
import scipy.sparse as sp
import torch

import sparsepoly_b200 as S
from sparsepoly_b200 import _lib, dataset, kernels, multi, synth

pytestmark = pytest.mark.gpu

FM_R, FM_C = S.SparseFactorizationMachineRegressor, S.SparseFactorizationMachineClassifier
AS_R, AS_C = S.SparseAllSubsetsRegressor, S.SparseAllSubsetsClassifier
NO_ROW = 2 ** 63 - 1
PSGD = dict(solver="psgd", max_iter=3, tol=-1.0, n_iter_no_change=10 ** 9, batch_size=16, eta0=0.05)


@pytest.fixture(autouse=True)
def _quiet(recwarn):
    yield                                             # convergence warnings of the short fits are expected


def cuda_csr(X, index=torch.int32, value=torch.float64):
    """The CUDA sparse CSR tensor of scipy matrix X, arrays as they are (unsorted rows and duplicates kept)."""
    X = X if sp.isspmatrix_csr(X) else sp.csr_matrix(X)
    t = lambda a, dt: torch.from_numpy(np.asarray(a)).to(dt)              # noqa: E731
    return torch.sparse_csr_tensor(t(X.indptr, index), t(X.indices, index), t(X.data, value), size=X.shape,
                                   device="cuda")


def _data(n=90, d=16, seed=0):
    X = synth.uniform_sparse(n, d, 5, seed)
    rng = np.random.RandomState(seed)
    return X, rng.randn(n), (rng.rand(n) < 0.4).astype(np.int64)


def _state(est):
    return {k: getattr(est, k) for k in ("P_", "w_", "lams_", "n_iter_", "it_") if hasattr(est, k)}


def _same(a, b):
    assert a.keys() == b.keys()
    for k in a:
        assert np.array_equal(np.asarray(a[k]), np.asarray(b[k])), k


def _host_csr_equal(dcsr, X_host):
    want = dataset.host_csr(X_host)
    got = [t.cpu().numpy() for t in (dcsr.indptr, dcsr.indices, dcsr.data)]
    for g, w in zip(got, want):
        assert g.dtype == w.dtype and np.array_equal(g, w)


# ------------------------------------------------------------------ every estimator, solver and fit_lower
FIT_CASES = [
    ("fm_pcd_sql12", FM_R, dict(solver="pcd", regularizer="squaredl12", degree=2, max_iter=4)),
    ("fm_pcd_omegati_d3", FM_C, dict(solver="pcd", regularizer="omegati", degree=3, loss="logistic", max_iter=4)),
    ("fm_pbcd_l21_d3", FM_C, dict(solver="pbcd", regularizer="l21", degree=3, max_iter=4)),
    ("fm_pbcd_sql21_none", FM_R, dict(solver="pbcd", regularizer="squaredl21", degree=2, fit_lower=None, max_iter=4)),
    ("fm_psgd_l1_planned", FM_C, dict(PSGD, regularizer="l1", degree=2, loss="logistic")),
    ("fm_psgd_sql12_planned", FM_R, dict(PSGD, regularizer="squaredl12", degree=2)),
    ("fm_psgd_l21_dense_grad", FM_R, dict(PSGD, regularizer="l21", degree=3)),
    ("fm_psgd_sql21_dense_grad_clf", FM_C, dict(PSGD, regularizer="squaredl21", degree=2, batch_size="auto")),
    ("as_pcd", AS_R, dict(solver="pcd", regularizer="omegati", max_iter=4)),
    ("as_pbcd_clf", AS_C, dict(solver="pbcd", regularizer="l1", max_iter=4)),
] + [(f"fm_augment_d{m}_{lin}", FM_R, dict(solver="pcd", regularizer="l1", degree=m, fit_lower="augment",
                                             fit_linear=lin == "lin", max_iter=3))
     for m in (2, 3, 4, 5) for lin in ("lin", "nolin")] + [
    ("fm_augment_psgd_d4", FM_C, dict(PSGD, regularizer="l1", degree=4, fit_lower="augment")),
    ("fm_augment_pbcd_d3", FM_R, dict(solver="pbcd", regularizer="l1", degree=3, fit_lower="augment", max_iter=3)),
]


@pytest.mark.parametrize("tag,cls,kw", FIT_CASES, ids=[c[0] for c in FIT_CASES])
def test_fit_predict_objective_match_host(tag, cls, kw):
    X, yr, yc = _data(seed=len(tag))
    y = yc if cls in (FM_C, AS_C) else yr
    _host_csr_equal(dataset.check_X(cuda_csr(X)), X)
    host = cls(random_state=0, **kw).fit(X, y)
    dev = cls(random_state=0, **kw).fit(cuda_csr(X), torch.from_numpy(y).cuda())     # y on the device too
    if kw["solver"] == "psgd" and kw["regularizer"] in ("l21", "squaredl21"):
        # the dense-gradient path sums its gradients with fp64 atomics: not bit-reproducible even between two host fits
        for k, v in _state(host).items():
            assert np.allclose(v, _state(dev)[k], rtol=1e-9, atol=1e-15), k
    else:
        _same(_state(host), _state(dev))
    Xte = synth.uniform_sparse(40, X.shape[1], 6, 99)
    Xte_d = cuda_csr(Xte)
    for est in (host, dev):                             # the same model on host X and on device X
        if cls in (FM_C, AS_C):
            assert np.array_equal(est.decision_function(Xte), est.decision_function(Xte_d))
            assert np.array_equal(est.predict(Xte), est.predict(Xte_d))
            if kw.get("loss") == "logistic":
                assert np.array_equal(est.predict_proba(Xte), est.predict_proba(Xte_d))
        else:
            assert np.array_equal(est.predict(Xte), est.predict(Xte_d))
        assert S.objective(est, X, y) == S.objective(est, cuda_csr(X), torch.from_numpy(y))


# ------------------------------------------------------------------ input variants against the host path
def _noncanonical(n=60, d=20, seed=3):
    """Rows with unsorted columns, at most two entries per (row, column), explicit zeros and a pair summing to 0."""
    rng = np.random.RandomState(seed)
    indptr, indices, data = [0], [], []
    for i in range(n):
        cols = list(rng.choice(d, rng.randint(0, 8), replace=False))
        cols += list(rng.choice(cols, min(len(cols), rng.randint(0, 3)), replace=False)) if cols else []
        rng.shuffle(cols)
        vals = list(rng.randn(len(cols)))
        if i % 7 == 0 and cols:
            vals[0] = 0.0                                    # explicit zero
        if i % 5 == 0 and cols and cols.count(cols[0]) == 1:
            cols.append(cols[0])                             # a duplicate pair that sums to zero (kept stored)
            vals.append(-vals[0])
        indices += cols
        data += vals
        indptr.append(len(indices))
    return sp.csr_matrix((np.array(data), np.array(indices, dtype=np.int32), np.array(indptr, dtype=np.int32)),
                         shape=(n, d))


def _variants():
    X, _, _ = _data(n=70, d=18, seed=5)
    long_row = sp.random(5, 3000, density=0.0, format="lil")
    long_row[2, np.arange(0, 3000, 3)] = np.arange(1, 1001) / 7.0       # one row of 1000 entries: > a 256-thread block
    long_row = sp.vstack([long_row.tocsr(), synth.uniform_sparse(20, 3000, 4, 8)]).tocsr()
    empty = X.tolil()
    empty[[0, 5, 69], :] = 0
    empty = empty.tocsr()
    empty.eliminate_zeros()
    A = X.toarray() + 0.25 * np.random.RandomState(6).randn(*X.shape)
    At = torch.from_numpy(np.ascontiguousarray(A.T)).cuda()
    Xnc = _noncanonical()
    assert not Xnc.has_canonical_format
    return [
        ("int64", X, cuda_csr(X, torch.int64)),
        ("int64_float32", X.astype(np.float32), cuda_csr(X.astype(np.float32), torch.int64, torch.float32)),
        ("float32", X.astype(np.float32), cuda_csr(X.astype(np.float32), value=torch.float32)),
        ("dense", A, torch.from_numpy(A).cuda()),
        ("dense_float32", A.astype(np.float32), torch.from_numpy(A.astype(np.float32)).cuda()),
        ("dense_transposed_view", A, At.T),
        ("noncanonical", Xnc, cuda_csr(Xnc)),
        ("noncanonical_int64_float32", Xnc.astype(np.float32), cuda_csr(Xnc.astype(np.float32), torch.int64,
                                                                        torch.float32)),
        ("empty_rows", empty, cuda_csr(empty)),
        ("long_row", long_row, cuda_csr(long_row)),
    ]


@pytest.mark.parametrize("i", range(10), ids=["int64", "int64_float32", "float32", "dense", "dense_float32",
                                          "dense_transposed_view", "noncanonical", "noncanonical_int64_float32",
                                          "empty_rows", "long_row"])
def test_input_variants_match_host(i):
    tag, Xh, Xd = _variants()[i]
    _host_csr_equal(dataset.check_X(Xd), Xh)
    y = np.random.RandomState(i).randn(Xh.shape[0])
    for kw in (dict(solver="pcd", regularizer="squaredl12", max_iter=3),
               dict(PSGD, regularizer="l1", batch_size="auto"),
               dict(solver="pbcd", regularizer="l1", degree=3, fit_lower="augment", max_iter=2)):
        host = FM_R(random_state=1, **kw).fit(Xh, y)
        dev = FM_R(random_state=1, **kw).fit(Xd, y)
        _same(_state(host), _state(dev))
        assert np.array_equal(host.predict(Xh), dev.predict(Xd))
    P = np.random.RandomState(2).randn(3, Xh.shape[1])
    assert np.array_equal(kernels.anova_kernel(Xh, P, 3), kernels.anova_kernel(Xd, P, 3))
    assert np.array_equal(kernels.all_subsets_kernel(Xh, P), kernels.all_subsets_kernel(Xd, P))
    lams = np.array([1.0, -1.0, 1.0])
    assert np.array_equal(kernels.poly_predict(Xh, P, lams, "poly", 2), kernels.poly_predict(Xd, P, lams, "poly", 2))


def test_augmented_layout_matches_add_dummy_feature():
    from sklearn.preprocessing import add_dummy_feature
    X = _noncanonical(seed=11)
    for n_dummy in (1, 2, 3, 4):
        Xh = X
        for _ in range(n_dummy):
            Xh = add_dummy_feature(Xh, value=1)
        _host_csr_equal(dataset.check_X(cuda_csr(X)).augment(n_dummy), Xh)


# ------------------------------------------------------------------ the check kernel's report
def _np_report(indptr, indices, values, n_cols):
    """sp_csr_prepare's report restated (include/sparsepoly_b200.h)."""
    n, nnz = len(indptr) - 1, len(values)
    r = [NO_ROW, int(indptr[0]), int(indptr[n]), NO_ROW, NO_ROW, NO_ROW, 0, NO_ROW]
    for i in range(n):
        a, b = int(indptr[i]), int(indptr[i + 1])
        if b < a:
            r[0] = min(r[0], i)
        s = min(max(a, 0), nnz)
        e = min(max(b, s), nnz)
        c, v = indices[s:e].astype(np.int64), values[s:e].astype(np.float64)
        if np.any((c < 0) | (c >= n_cols)):
            r[3] = min(r[3], i)
        if np.any(np.isnan(v)):
            r[4] = min(r[4], i)
        if np.any(np.isinf(v)):
            r[5] = min(r[5], i)
        if np.any(np.diff(c) <= 0):
            r[6] += 1
            r[7] = min(r[7], i)
    return r


def _faulty(kind, row, itype, vtype, seed):
    X = sp.vstack([synth.uniform_sparse(150, 400, 6, seed), sp.csr_matrix(np.ones((1, 400))),
                   synth.uniform_sparse(149, 400, 6, seed + 1)]).tocsr()              # row 150: 400 entries
    indptr, indices, data = X.indptr.astype(itype), X.indices.astype(itype), X.data.astype(vtype)
    s, e = int(indptr[row]), int(indptr[row + 1])
    if kind == "range":
        indices[e - 1] = 400 if seed % 2 else -1
    elif kind == "nan":
        data[e - 1] = np.nan
    elif kind == "inf":
        data[s] = -np.inf
    elif kind == "unsorted":
        indices[s], indices[e - 1] = indices[e - 1], indices[s]
    elif kind == "duplicate":
        indices[e - 1] = indices[e - 2]
    elif kind == "decreasing":
        indptr[row + 1] = indptr[row] - 1
    elif kind == "indptr_ends":
        indptr[0], indptr[-1] = 1, indptr[-1] - 2
    return indptr, indices, data


@pytest.mark.parametrize("kind", ["none", "range", "nan", "inf", "unsorted", "duplicate", "decreasing",
                                  "indptr_ends"])
@pytest.mark.parametrize("row", [0, 150, 299])
@pytest.mark.parametrize("itype,vtype", [(np.int32, np.float64), (np.int64, np.float32)])
def test_check_report_matches_numpy(kind, row, itype, vtype):
    indptr, indices, data = _faulty(kind, row, itype, vtype, seed=row + len(kind))
    t = lambda a: torch.from_numpy(a).cuda()                              # noqa: E731
    for out in (False, True):
        o = dataset._alloc_csr(300, len(data), torch.device("cuda")) if out else None
        rep = dataset._run_prepare(300, 400, t(indptr), t(indices), t(data), (0, 0), 0, o).tolist()
        assert rep == _np_report(indptr, indices, data, 400), (kind, row, out)


def test_dense_report_and_layout():
    A = np.random.RandomState(0).randn(40, 300)
    A[0, 5], A[17, 299], A[39, 0], A[39, 1] = np.inf, np.nan, np.nan, -np.inf
    Ad = torch.from_numpy(A).cuda()
    rep = dataset._run_prepare(40, 300, None, None, Ad, Ad.stride(), 0).tolist()
    assert rep == [NO_ROW, 0, 40 * 300, NO_ROW, 17, 0, 0, NO_ROW]


# ------------------------------------------------------------------ errors: raised before the estimator changes
def _bad_inputs():
    X, _, _ = _data()
    t = lambda a, dt=torch.int32: torch.from_numpy(np.asarray(a)).to(dt).cuda()   # noqa: E731
    ip, ix, v = X.indptr.copy(), X.indices.copy(), X.data.copy()

    def csr(ip_, ix_, v_, shape=X.shape, dt=torch.float64):
        return torch.sparse_csr_tensor(t(ip_), t(ix_), t(v_, dt), size=shape)
    v_nan, v_inf = v.copy(), v.copy()
    v_nan[ip[4]] = np.nan
    v_inf[ip[7]] = np.inf
    ix_bad = ix.copy()
    ix_bad[ip[3]] = X.shape[1]
    ip_dec = ip.copy()
    ip_dec[10] = ip[11] + 1
    ip_end = ip.copy()
    ip_end[-1] -= 1
    ip0 = ip.copy()
    ip0[0] = 1
    return [
        ("nan", csr(ip, ix, v_nan), "contains NaN. First in row 4"),
        ("inf", csr(ip, ix, v_inf), "contains infinity or a value too large for dtype\\('float64'\\). First in row 7"),
        ("range", csr(ip, ix_bad, v), "outside \\[0, 16\\) in row 3"),
        ("decreasing", csr(ip_dec, ix, v), "indptr decreases at row 10"),
        ("indptr_end", csr(ip_end, ix, v), "indptr\\[-1\\]"),
        ("indptr0", csr(ip0, ix, v), "indptr\\[0\\] is 1"),
        ("coo", torch.from_numpy(X.toarray()).cuda().to_sparse(), "layout"),
        ("float16", csr(ip, ix, v, dt=torch.float16), "float32 or float64"),
        ("int_dense", torch.ones(X.shape, dtype=torch.int64, device="cuda"), "float32 or float64"),
        ("3d", torch.ones((2, 3, 4), dtype=torch.float64, device="cuda"), "2-D"),
        ("batched_csr", torch.ones((2, 3, 4), dtype=torch.float64, device="cuda").to_sparse_csr(), "2-D"),
        ("no_rows", torch.sparse_csr_tensor(t([0]), t([]), t([], torch.float64), size=(0, 16)),
         "Found array with 0 sample\\(s\\) \\(shape=\\(0, 16\\)\\) while a minimum of 1 is required."),
    ]


@pytest.mark.parametrize("i", range(12))
@pytest.mark.parametrize("cls,kw", [(FM_R, dict(solver="pcd")), (FM_C, dict(solver="psgd", regularizer="l1")),
                                    (AS_R, dict(solver="pbcd", regularizer="l1"))])
def test_errors_leave_the_estimator_unfitted(i, cls, kw):
    tag, Xbad, match = _bad_inputs()[i]
    y = np.arange(90) % 2
    est = cls(**kw)
    with pytest.raises(ValueError, match=match):
        est.fit(Xbad, y)
    assert not hasattr(est, "P_")
    if tag == "nan":                                   # check_X_y's wording at the regressor's site, check_array's at
        with pytest.raises(ValueError, match="Input X contains NaN" if cls is not FM_C else "Input contains NaN"):
            cls(**kw).fit(Xbad, y)                     # the classifier's binary fast path: as the host path
    if cls is FM_C:
        with pytest.raises(ValueError, match=match):
            est.partial_fit(Xbad, y, classes=[0, 1])
        assert not hasattr(est, "P_") and not hasattr(est, "_psgd_stream")


def test_wrong_device_is_named():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    X, y, _ = _data()
    Xd = cuda_csr(X).to("cuda:1")
    est = FM_R()
    with pytest.raises(ValueError, match="cuda:1.*cuda:0"):
        est.fit(Xd, y)
    assert not hasattr(est, "P_")


# ------------------------------------------------------------------ zero copy
def test_canonical_input_is_wrapped_and_never_written():
    X, y, yc = _data(n=200, d=30, seed=4)
    Xd = cuda_csr(X)
    before = [t.clone() for t in (Xd.crow_indices(), Xd.col_indices(), Xd.values())]
    dc = dataset.check_X(Xd)
    assert [a.data_ptr() for a in (dc.indptr, dc.indices, dc.data)] == \
        [a.data_ptr() for a in (Xd.crow_indices(), Xd.col_indices(), Xd.values())]
    est = FM_R(solver="pcd", max_iter=2).fit(Xd, y)
    assert est._dev_state["ds"].csr[0].data_ptr() == Xd.crow_indices().data_ptr()
    assert est._h2d_bytes == y.nbytes + est.P_.nbytes + est.w_.nbytes
    clf = FM_C(**dict(PSGD, regularizer="squaredl12"))
    clf.fit(Xd, yc)
    assert clf._h2d_bytes == yc.astype(np.float64).nbytes + clf.P_.nbytes + clf.w_.nbytes
    for _ in range(2):
        clf.partial_fit(Xd, yc, classes=[0, 1])
    for b, a in zip(before, (Xd.crow_indices(), Xd.col_indices(), Xd.values())):
        assert torch.equal(a, b)
    Xn = cuda_csr(_noncanonical(), torch.int64, torch.float32)
    before = [t.clone() for t in (Xn.crow_indices(), Xn.col_indices(), Xn.values())]
    FM_R(solver="pcd", max_iter=2).fit(Xn, np.ones(Xn.shape[0]))
    for b, a in zip(before, (Xn.crow_indices(), Xn.col_indices(), Xn.values())):
        assert torch.equal(a, b)


# ------------------------------------------------------------------ partial_fit stream
@pytest.mark.parametrize("reg", ["l1", "squaredl12"])      # (the planned path: bit-reproducible, unlike l21's atomics)
def test_partial_fit_stream_matches_host(reg):
    X, _, yc = _data(n=256, d=40, seed=7)
    host = FM_C(**dict(PSGD, regularizer=reg, random_state=3))
    dev = FM_C(**dict(PSGD, regularizer=reg, random_state=3))
    for epoch in range(2):
        for c0 in range(0, 256, 64):
            host.partial_fit(X[c0:c0 + 64], yc[c0:c0 + 64], classes=[0, 1])
            dev.partial_fit(cuda_csr(X[c0:c0 + 64]), torch.from_numpy(yc[c0:c0 + 64]).cuda(), classes=[0, 1])
            _same(_state(host), _state(dev))
    assert dev._partial_fit_stats["rows"] == 64


# ------------------------------------------------------------------ many models
@pytest.mark.parametrize("solver,reg", [("pcd", "l1"), ("pbcd", "l21")])
def test_fit_many_and_scoring_many_match_host(solver, reg):
    X, y, _ = _data(n=120, d=20, seed=9)
    Y = [y, -y, 2 * y]

    def make():
        return [FM_R(solver=solver, regularizer=reg, degree=3, gamma=g, max_iter=3, fit_lower="augment",
                     random_state=i) for i, g in enumerate((0.1, 1.0, 3.0))]
    host, dev = multi.fit_many(make(), X, Y), multi.fit_many(make(), cuda_csr(X), [torch.from_numpy(t) for t in Y])
    for h, d in zip(host, dev):
        _same(_state(h), _state(d))
    Xte = synth.uniform_sparse(30, 20, 5, 10)
    yte = np.random.RandomState(1).randn(30)
    for Xh, Xd in ((Xte, cuda_csr(Xte)), (Xte.toarray(), torch.from_numpy(Xte.toarray()).cuda())):
        assert np.array_equal(S.decision_function_many(host, Xh), S.decision_function_many(dev, Xd))
        assert np.array_equal(S.predict_many(host, Xh), S.predict_many(dev, Xd))
        assert np.array_equal(S.score_many(host, Xh, yte), S.score_many(dev, Xd, torch.from_numpy(yte).cuda()))
        assert S.objective_many(host, Xh, yte) == S.objective_many(dev, Xd, torch.from_numpy(yte))
    empty = torch.sparse_csr_tensor(torch.zeros(1, dtype=torch.int32), torch.zeros(0, dtype=torch.int32),
                                    torch.zeros(0, dtype=torch.float64), size=(0, 20), device="cuda")
    assert S.decision_function_many(dev, empty).shape == (3, 0)
    assert np.array_equal(S.predict_many(host, sp.csr_matrix((0, 20))), S.predict_many(dev, empty))
    assert S.objective_many(host, sp.csr_matrix((0, 20)), np.zeros(0)) == S.objective_many(dev, empty, np.zeros(0))


def test_anova_kernel_matches_host():
    X, _, _ = _data(n=50, d=25, seed=12)
    P = np.random.RandomState(0).randn(4, 25)
    for m in (2, 3, 4, 5):
        assert np.array_equal(kernels.anova_kernel(X, P, m), kernels.anova_kernel(cuda_csr(X, torch.int64), P, m))


# ------------------------------------------------------------------ sharded psgd with device shards
def _sharded_worker(rank, world, port, out_dir, n_dev):
    import sys
    import torch.distributed as dist
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank % n_dev)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    import sparsepoly_b200 as S_
    from sparsepoly_b200 import distributed
    distributed.enable_sharding()
    X = synth.criteo_like(1500, 600, 21 + rank)
    y = np.where(np.random.RandomState(31 + rank).rand(1500) < 0.3, 1.0, -1.0)
    Xte = synth.criteo_like(40 + 10 * rank, 600, 77 + rank)
    res = {}
    for tag, (Xr, yr, Xt) in (("host", (X, y, Xte)), ("dev", (cuda_csr(X), torch.from_numpy(y).cuda(), cuda_csr(Xte)))):
        est = S_.SparseFactorizationMachineClassifier(random_state=rank, **dict(PSGD, regularizer="squaredl12",
                                                                                 loss="logistic", batch_size=256))
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            est.fit(Xr, yr)
        res[tag + "/P"], res[tag + "/w"] = est.P_, est.w_
        res[tag + "/pred"] = distributed.sharded_predict(est, Xt)
    np.savez(os.path.join(out_dir, f"rank{rank}.npz"), **res)
    dist.barrier()
    dist.destroy_process_group()


def test_sharded_psgd_with_device_shards_matches_host_shards(tmp_path):
    import torch.multiprocessing as mp
    world = 2
    if torch.cuda.device_count() < world:
        pytest.skip("needs one GPU per rank")
    port = 35600 + (os.getpid() % 2000)
    mp.spawn(_sharded_worker, args=(world, port, str(tmp_path), torch.cuda.device_count()), nprocs=world, join=True)
    for r in range(world):
        z = np.load(tmp_path / f"rank{r}.npz")
        for k in ("P", "w", "pred"):
            assert np.array_equal(z["host/" + k], z["dev/" + k]), (r, k)
