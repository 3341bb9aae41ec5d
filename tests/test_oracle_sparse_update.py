"""oracle.sparse_update (the method of kr_trace_fun_sparse_update) against dense truth: tr f(Ã) - tr f(Ã - D) from
eigvalsh on both matrices, 1e-10 relative of the difference, on Anaheim, two power grids and Oregon A0 for exp, sinh and
cosh, with Ω holding edges, non-edges and diagonal pairs; X = 0 gives exactly 0; and the chosen quadrature order meets
its error bound where two orders fewer visibly do not."""
import math

import numpy as np
import pytest
import scipy.sparse as sp
from scipy.linalg import eigh

from conftest import load_graph

F = {"exp": np.exp, "sinh": np.sinh, "cosh": np.cosh}
DF = {"exp": np.exp, "sinh": np.cosh, "cosh": np.sinh}


def case(name, seed=1, m=30):
    """A / max(A), Ω = m random edges (X in [-0.5 a_ij, 0]: weights lowered, some removed almost entirely) plus two
    non-edges and two diagonal pairs; returns Ã = A + Δ(X, Ω), X, Ω."""
    import oracle.sparse_update as S
    A = sp.csr_matrix(load_graph(name)).astype(np.float64)
    A = (A / A.max()).tocsr()
    n = A.shape[0]
    rng = np.random.default_rng(seed)
    L = sp.tril(A, -1).tocoo()
    pick = rng.choice(L.nnz, m, replace=False)
    Om = np.stack([L.row[pick] + 1, L.col[pick] + 1], 1)
    X = -0.5 * L.data[pick] * rng.random(m)
    extra = [[1, n], [5, n - 3], [7, 7], [n // 2, n // 2]]
    assert A[0, n - 1] == 0 and A[4, n - 4] == 0
    Om = np.vstack([Om, extra]).astype(np.int64)
    X = np.concatenate([X, [0.3, 0.2, 0.25, -0.1]])
    return (A + S.delta(X, Om, n)).tocsr(), X, Om


def tol_for(At, fun):
    import oracle as O
    return 1e-14 * np.cosh(O.normest(At, 1e-2)[0])


@pytest.mark.parametrize("name", ["transport_Anaheim", "grid_England", "grid_Mexico", "oregon_A0"])
@pytest.mark.parametrize("fun", ["exp", "sinh", "cosh"])
def test_oracle_matches_dense_truth(name, fun):
    import oracle.sparse_update as S
    At, X, Om = case(name)
    D = S.delta(X, Om, At.shape[0]).toarray()
    truth = F[fun](np.linalg.eigvalsh(At.toarray())).sum() - F[fun](np.linalg.eigvalsh(At.toarray() - D)).sum()
    dtr, q, it = S.trace_fun_sparse_update(At, X, Om, fun, tol_for(At, fun), 100)
    assert abs(dtr - truth) <= 1e-10 * abs(truth), (dtr, truth)
    assert 1 <= q <= 32 and 3 < it <= 100


def test_zero_direction_is_exactly_zero():
    import oracle.sparse_update as S
    At, X, Om = case("transport_Anaheim")
    assert S.trace_fun_sparse_update(At, 0 * X, Om, "sinh", 1e-10, 100) == (0.0, 0, 0)


def test_duplicate_and_mirrored_pairs_add_up():
    # (i, j) twice and (j, i) once: D(i, j) is the sum of the three values, as sparse() assembles it
    import oracle.sparse_update as S
    At, X, Om = case("grid_England", m=10)
    i, j = Om[0]
    Om2 = np.vstack([Om, [[i, j], [j, i]]])
    X2 = np.concatenate([X, [0.05, -0.02]])
    Xs = X.copy()
    Xs[0] += 0.03
    a = S.trace_fun_sparse_update(At, X2, Om2, "exp", 1e-12, 100)[0]
    b = S.trace_fun_sparse_update(At, Xs, Om, "exp", 1e-12, 100)[0]
    assert abs(a - b) <= 1e-10 * abs(b)


@pytest.mark.parametrize("fun", ["exp", "sinh", "cosh"])
def test_chosen_order_meets_the_bound(fun):
    """The quadrature alone (exact integrand from eigh): at the chosen q its error is within the bound and within
    tol * sum c|X|; at q - 2 it is far above that target - the bound is not loose on a 3 x 3 case."""
    import oracle.sparse_update as S
    At = np.array([[2.0, 1.0, 0.0], [1.0, 0.0, 1.0], [0.0, 1.0, 0.0]])
    Om = np.array([[1, 1], [1, 2]])
    X = np.array([2.0, 0.5])
    D = S.delta(X, Om, 3).toarray()
    cx = np.array([1.0, 2.0]) * X
    truth = F[fun](np.linalg.eigvalsh(At)).sum() - F[fun](np.linalg.eigvalsh(At - D)).sum()

    def quad(q):
        t, w = S.gauss_legendre01(q)
        s = 0.0
        for ti, wi in zip(t, w):
            lam, V = eigh(At - (1 - ti) * D)
            Fp = (V * DF[fun](lam)) @ V.T
            s += wi * float(np.dot(cx, Fp[Om[:, 0] - 1, Om[:, 1] - 1]))
        return s

    nD, nA = float(np.abs(D).sum(1).max()), float(np.linalg.norm(At, 2))
    tol = 1e-8
    target = tol * np.abs(cx).sum()
    q = S.choose_q(3, nD, nA, tol, np.abs(cx).sum())
    bound = math.exp(S.log_error_bound(q, 3, nD, nA))
    assert bound <= target < math.exp(S.log_error_bound(q - 1, 3, nD, nA))
    assert abs(quad(q) - truth) <= bound
    assert abs(quad(q - 2) - truth) > 10 * target
    # and through the entries of the oracle's Krylov spaces
    dtr = S.trace_fun_sparse_update(sp.csr_matrix(At), X, Om, fun, tol, 3)[0]
    assert abs(dtr - truth) <= target


def test_order_cap_and_qmax():
    import oracle.sparse_update as S
    assert S.choose_q(100, 1.0, 1.0, 0.0, 1.0) == 32
    assert S.choose_q(100, 1.0, 1.0, 0.0, 1.0, qmax=5) == 5
    assert S.choose_q(100, 0.0, 1.0, 1e-12, 1.0) == 1
    t, w = S.gauss_legendre01(7)
    assert abs(w.sum() - 1.0) < 1e-15 and np.all(np.diff(t) > 0)


def test_oracle_matches_reference_golden_objective():
    """Anaheim, Ω = all 634 edges, f = sinh: -dtr against the objective slice of the reference's literal call, at the
    tolerance the sparse gradient is checked with (tests/test_reference_goldens.py)."""
    import json
    import os
    import warnings
    import scipy.io as sio
    import oracle as O
    import oracle.sparse_update as S
    from conftest import GOLDEN
    ref = json.load(open(os.path.join(GOLDEN, "reference_golden.json")))["Anaheim_all_edges_fg_sinh"]
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        I = sio.loadmat(os.path.join(GOLDEN, "reference_inputs.mat"))
    An = sp.csr_matrix(I["Anaheim"])
    Om, X = I["Anaheim_Omega"].astype(np.int64), I["Anaheim_X"].ravel()
    At = (An + S.delta(X, Om, An.shape[0])).tocsr()
    tol = 1e-10 * np.cosh(float(O.normest(An, 1e-6)[0]))
    dtr = S.trace_fun_sparse_update(At, X, Om, "sinh", tol, 100)[0]
    assert abs(-dtr - ref[0]) <= 1e-9 * abs(ref[0]), (-dtr, ref[0])
