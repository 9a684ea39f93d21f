"""An exact reference for the kernel values, independent of the C oracle and of CUDA, and the oracle's
kernels checked against it at every supported degree.

Every fp64 input is a dyadic rational, so the ANOVA / all-subsets dynamic programs run exactly in Python
integers scaled by a common power of two.  The same recurrence on |x|*|p| (`abs_ref`) bounds what the fp64
evaluation may lose to rounding:

    |K - exact| <= c * (nnz_row + m) * 2^-53 * abs_ref

With signed P the terms cancel and the elementwise relative error of a correct fp64 DP reaches 1e-13, so a
fixed relative tolerance would be either vacuous or flaky; this bound is neither.  The oracle's
`anova_kernel` uses the power-sum (Newton-Girard) form of the reference instead of the DP; it is held to
the same bound computed from that form's own absolute-value recurrence, which is looser wherever one
|x_j p_j| dominates a row.

tests/test_kernel_variants_gpu.py uses the same reference for the CUDA row kernels."""
import itertools
import math
from fractions import Fraction

import numpy as np
import pytest
import scipy.sparse as sp

from oracle import oracle as O

EPS = 2.0 ** -53
C_BOUND = 4
DEGREES = [1, 2, 3, 4, 5, -1]
ROW_NNZ = (0, 1, 7, 8, 9, 31, 32, 33, 200)


# ------------------------------------------------------------------------------------------ exact reference
def _dyadic(a):
    """a (float array) -> (numerators, exponents) with a == num / 2**e exactly (num: Python ints)."""
    a = np.asarray(a, dtype=np.float64)
    num = np.empty(a.shape, dtype=object)
    ex = np.empty(a.shape, dtype=np.int64)
    for idx, v in np.ndenumerate(a):
        n, den = float(v).as_integer_ratio()
        num[idx] = n
        ex[idx] = den.bit_length() - 1
    return num, ex


def _row_terms(X, P_num, P_ex, i):
    """x_j * p_j[s] of row i as Python ints over the common scale 2**S: (v [nnz, k] object, S)."""
    st, en = X.indptr[i], X.indptr[i + 1]
    cols = X.indices[st:en]
    x_num, x_ex = _dyadic(X.data[st:en])
    num = x_num[:, None] * P_num[cols]
    ex = x_ex[:, None] + P_ex[cols]
    S = int(ex.max()) if ex.size else 0
    scale = np.array([1 << int(S - e) for e in ex.ravel()], dtype=object).reshape(ex.shape)
    return num * scale, S


def _csr(X):
    X = sp.csr_matrix(X, dtype=np.float64)
    X.sum_duplicates()
    X.sort_indices()
    return X


def exact_anova_degrees(X, P_dk, max_degree=5):
    """{m: (K, abs_ref)} for m = 1..max_degree: the ANOVA kernel K[i, s] = e_m(x_j p_j[s] : j in row i) and
    the same elementary symmetric polynomial of |x_j p_j[s]|, both exact and then rounded once to fp64."""
    X = _csr(X)
    P_num, P_ex = _dyadic(P_dk)
    n, k = X.shape[0], P_dk.shape[1]
    out = {m: (np.zeros((n, k)), np.zeros((n, k))) for m in range(1, max_degree + 1)}
    for i in range(n):
        v, S = _row_terms(X, P_num, P_ex, i)
        va = np.abs(v)
        A = [np.ones(k, dtype=object)] + [np.zeros(k, dtype=object) for _ in range(max_degree)]
        B = [np.ones(k, dtype=object)] + [np.zeros(k, dtype=object) for _ in range(max_degree)]
        for q in range(v.shape[0]):
            for t in range(max_degree, 0, -1):
                A[t] = A[t] + A[t - 1] * v[q]
                B[t] = B[t] + B[t - 1] * va[q]
        for m in range(1, max_degree + 1):
            den = 1 << (S * m)
            out[m][0][i] = [float(Fraction(int(a), den)) for a in A[m]]
            out[m][1][i] = [float(Fraction(int(b), den)) for b in B[m]]
    return out


def exact_anova(X, P_dk, m):
    """(K, abs_ref) of the degree-m ANOVA kernel, P_dk [d, k]."""
    return exact_anova_degrees(X, P_dk, m)[m]


def exact_all_subsets(X, P_dk):
    """(K, abs_ref) of the all-subsets kernel prod_j (1 + x_j p_j[s]) and of prod_j (1 + |x_j p_j[s]|)."""
    X = _csr(X)
    P_num, P_ex = _dyadic(P_dk)
    n, k = X.shape[0], P_dk.shape[1]
    K, Kabs = np.ones((n, k)), np.ones((n, k))
    for i in range(n):
        v, S = _row_terms(X, P_num, P_ex, i)
        one = 1 << S
        A = np.ones(k, dtype=object)
        B = np.ones(k, dtype=object)
        for q in range(v.shape[0]):
            A = A * (one + v[q])
            B = B * (one + np.abs(v[q]))
        den = 1 << (S * v.shape[0])
        K[i] = [float(Fraction(int(a), den)) for a in A]
        Kabs[i] = [float(Fraction(int(b), den)) for b in B]
    return K, Kabs


def exact_kernel(X, P_dk, degree):
    return exact_all_subsets(X, P_dk) if degree == -1 else exact_anova(X, P_dk, degree)


def dp_bound(X, abs_ref, degree, c=C_BOUND):
    """Rounding bound of the fp64 DP on row i: c * (nnz_i + m) * 2^-53 * abs_ref[i, s]."""
    nnz = np.diff(_csr(X).indptr)[:, None]
    m = 1 if degree == -1 else degree
    return c * (nnz + m) * EPS * abs_ref


def prediction_bound(X, abs_ref, lams, degree, c=C_BOUND, linear_abs=None):
    """Bound of sum_s lams[s] K[i, s] (+ <w, x_i>): the kernel bounds plus the rounding of the sums over
    the k components and the row's nonzeros."""
    k = abs_ref.shape[1]
    nnz = np.diff(_csr(X).indptr)
    terms = np.abs(lams)[None, :] * abs_ref
    b = dp_bound(X, terms, degree, c).sum(1) + c * k * EPS * terms.sum(1)
    if linear_abs is not None:
        b = b + c * (nnz + k) * EPS * linear_abs
    return b


def exact_prediction(K_exact, lams, linear=None):
    """sum_s lams[s] K_exact[i, s] (+ linear[i]), summed without rounding error beyond the final one."""
    out = np.array([math.fsum(np.asarray(lams) * row) for row in K_exact])
    return out if linear is None else out + linear


def exact_linear(X, w):
    """(<w, x_i> rounded once, sum_j |w_j x_ij|) per row."""
    X = _csr(X)
    val, ab = np.zeros(X.shape[0]), np.zeros(X.shape[0])
    for i in range(X.shape[0]):
        st, en = X.indptr[i], X.indptr[i + 1]
        terms = [Fraction(float(a)) * Fraction(float(b)) for a, b in zip(X.data[st:en], w[X.indices[st:en]])]
        val[i] = float(sum(terms, Fraction(0)))
        ab[i] = float(sum((abs(t) for t in terms), Fraction(0)))
    return val, ab


def assert_within(got, want, bound, what=""):
    got, want, bound = (np.asarray(a, dtype=np.float64) for a in (got, want, bound))
    err = np.abs(got - want)
    bad = ~(err <= bound)
    if np.any(bad):
        i = tuple(np.argwhere(bad)[0])
        raise AssertionError(f"{what}: |got - exact| = {err[i]:.3e} > bound {bound[i]:.3e} at {i} "
                             f"(got {got[i]!r}, exact {want[i]!r}); {int(bad.sum())} entries out of bound")


# ------------------------------------------------------------------------------------------ test inputs
def rows_matrix(d=400, lengths=ROW_NNZ, seed=0, big_row=True):
    """CSR with one row per entry of `lengths` (sorted, distinct columns, N(0,1) values) and, with big_row,
    a 9-nonzero row whose first value is 1e3 (|x p| ~ 1e3 against N(0,1) P)."""
    rng = np.random.RandomState(seed)
    indptr, indices, data = [0], [], []
    rows = [(r, None) for r in lengths] + ([(9, 1e3)] if big_row else [])
    for r, big in rows:
        cols = np.sort(rng.choice(d, r, replace=False))
        vals = rng.randn(r)
        if big is not None:
            vals[0] = big
        indices.extend(cols.tolist())
        data.extend(vals.tolist())
        indptr.append(len(indices))
    return sp.csr_matrix((np.array(data), np.array(indices, dtype=np.int32), np.array(indptr)),
                         shape=(len(rows), d))


def signed_P(d, k, seed, degree):
    """N(0,1) P_dk for the ANOVA kernels; for all-subsets scaled so that prod_j (1 + |x_j p_j|) over
    200 nonzeros stays finite (|x p| ~ 0.02)."""
    P = np.random.RandomState(seed).randn(d, k)
    return 0.02 * P if degree == -1 else P


# ------------------------------------------------------------------------------------------ tests
def test_exact_reference_matches_brute_force():
    """The exact DP against e_m by enumeration of subsets (Fractions), and prod_j (1 + x_j p_j)."""
    X = rows_matrix(d=30, lengths=(0, 1, 5, 8), seed=3, big_row=False)
    P = np.random.RandomState(4).randn(30, 3)
    Xc = _csr(X)
    ex = exact_anova_degrees(X, P, 5)
    Kall, Kall_abs = exact_all_subsets(X, P)
    for i in range(Xc.shape[0]):
        st, en = Xc.indptr[i], Xc.indptr[i + 1]
        for s in range(3):
            v = [Fraction(float(x)) * Fraction(float(P[j, s])) for x, j in zip(Xc.data[st:en], Xc.indices[st:en])]
            for m in range(1, 6):
                e = sum((math.prod(c) for c in itertools.combinations(v, m)), Fraction(0))
                ea = sum((math.prod(abs(t) for t in c) for c in itertools.combinations(v, m)), Fraction(0))
                assert ex[m][0][i, s] == float(e) and ex[m][1][i, s] == float(ea), (i, s, m)
            assert Kall[i, s] == float(math.prod((1 + t for t in v), start=Fraction(1)))
            assert Kall_abs[i, s] == float(math.prod((1 + abs(t) for t in v), start=Fraction(1)))


@pytest.mark.parametrize("degree", DEGREES)
def test_oracle_kernel_rows_dp_within_rounding_bound(degree):
    """sp_oracle_kernel_rows (the reference's DP, psgd.py:34-44 / kernels.py:118-129) on rows of 0..200
    nonzeros and one row with |x p| ~ 1e3, signed P."""
    X = rows_matrix()
    P = signed_P(X.shape[1], 5, 1, degree)
    want, abs_ref = exact_kernel(X, P, degree)
    got = O.kernel_rows_dp(X, P, degree)
    assert_within(got, want, dp_bound(X, abs_ref, degree), f"kernel_rows_dp degree {degree}")
    assert np.all(got[0] == (1.0 if degree == -1 else 0.0))            # the empty row is exact
    if degree == 5:
        assert np.max(np.abs(got - want)) <= 1e-14 * np.max(np.abs(want))


def _power_sum_abs(X, P_dk, degree):
    """Absolute-value recurrence of the power-sum form: a_m = (1/m) sum_t a_{m-t} p_t(|x p|)."""
    X = _csr(X)
    psums = [None] + [np.asarray(abs(X).power(t) @ (np.abs(P_dk) ** t)) for t in range(1, degree + 1)]
    a = [np.ones((X.shape[0], P_dk.shape[1]))]
    for m in range(1, degree + 1):
        a.append(sum(a[m - t] * psums[t] for t in range(1, m + 1)) / m)
    return a[degree]


@pytest.mark.parametrize("degree", DEGREES)
def test_oracle_kernels_and_poly_predict_within_rounding_bound(degree):
    """oracle.anova_kernel (power-sum form, kernels.py:71-115), all_subsets_kernel and poly_predict."""
    X = rows_matrix(seed=5)
    P = signed_P(X.shape[1], 6, 2, degree)
    lams = np.array([1.0, -1.0, 1.0, 1.0, -1.0, -1.0])
    want, abs_ref = exact_kernel(X, P, degree)
    if degree == -1:
        got = O.all_subsets_kernel(X, np.ascontiguousarray(P.T))
        bound_abs = abs_ref
        pred = O.poly_predict(X, np.ascontiguousarray(P.T), lams, "all-subsets")
    else:
        got = O.anova_kernel(X, np.ascontiguousarray(P.T), degree)
        bound_abs = _power_sum_abs(X, P, degree)
        assert np.all(bound_abs >= abs_ref * (1 - 1e-12))
        pred = O.poly_predict(X, np.ascontiguousarray(P.T), lams, "anova", degree)
    assert_within(got, want, dp_bound(X, bound_abs, degree), f"oracle kernel degree {degree}")
    assert_within(pred, exact_prediction(want, lams), prediction_bound(X, bound_abs, lams, degree),
                  f"oracle poly_predict degree {degree}")


@pytest.mark.parametrize("solver,reg,loss", [("pcd", "omegati", "squared"), ("pcd", "l1", "logistic"),
                                             ("pbcd", "omegacs", "squared"), ("pbcd", "l21", "squared_hinge")])
def test_oracle_degree5_objective_decreases(solver, reg, loss):
    """Degree-5 fits of the oracle (explicit lower orders): the objective after a short fit is below its
    value at the fit's starting point, as test_oracle_objective_decreases_on_reference_fits checks for the
    reference's own fits at degree <= 4."""
    from sklearn.utils import check_random_state
    from sparsepoly_b200 import synth
    n, d, k, degree = 400, 60, 3, 5
    X = synth.uniform_sparse(n, d, 8, 11)
    s = O.poly_predict(X, synth.planted_P(d, 3, 12, frac_features=0.3, scale=0.5), np.ones(3), "anova", 3)
    y = synth.targets_from_scores(s, 13, loss != "squared")
    common = dict(degree=degree, loss=loss, regularizer=reg, alpha=1e-3, beta=1e-3, gamma=1e-4, mean=True,
                  fit_lower="explicit", fit_linear=True)
    out = O.fit_fm(X, y, n_components=k, solver=solver, max_iter=3, tol=-1.0, random_state=0, **common)
    P0 = 0.01 * check_random_state(0).randn(degree - 1, k, d)
    start = O.objective_fm(X, y, P0, np.zeros(d), out["lams_"], **common)["total"]
    end = O.objective_fm(X, y, out["P_"], out["w_"], out["lams_"], **common)["total"]
    assert np.isfinite(end) and end < start, (start, end)
    assert 0.01 < np.mean(out["P_"] != 0) < 0.99
