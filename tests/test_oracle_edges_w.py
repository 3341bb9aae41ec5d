"""The per-candidate edge oracle (oracle.weighted_edges) against dense truth, and its greedy driver against the unweighted
oracle driver on a 0/1 graph.  Truth: sum f(eig(A + U B U')) - sum f(eig(A)) by eigvalsh, B = d_h [0 1; 1 0] (d_h on a
self loop)."""
import numpy as np
import pytest
import scipy.sparse as sp

from conftest import load_graph

import oracle as O
import oracle.weighted_edges as OW
from oracle.updates import _trace_formula

F = {"exp": np.exp, "sinh": np.sinh, "cosh": np.cosh}


def mixed_candidates(A, seed, n_edges=28, n_missing=8, n_loops=4):
    """Existing edges with d = -A(i, j) (weighted break), missing pairs with d in [0.5, 1.5] (weighted make) and self
    loops with d of either sign, shuffled: 40 candidates by default."""
    rng = np.random.default_rng(seed)
    n = A.shape[0]
    L = sp.tril(A, k=-1).tocoo()
    pick = rng.choice(L.nnz, n_edges, replace=False)
    E = [(int(L.row[p]) + 1, int(L.col[p]) + 1) for p in pick]
    d = [-float(L.data[p]) for p in pick]
    D = A.toarray()
    while len(E) < n_edges + n_missing:
        i, j = rng.choice(n, 2, replace=False)
        if D[i, j] == 0.0:
            E.append((int(i) + 1, int(j) + 1))
            d.append(float(rng.uniform(0.5, 1.5)))
    for v in rng.choice(n, n_loops, replace=False):
        E.append((int(v) + 1, int(v) + 1))
        d.append(float(rng.choice([-1.0, 1.0]) * rng.uniform(0.5, 1.5)))
    order = rng.permutation(len(E))
    return np.array(E, dtype=np.int64)[order], np.array(d)[order]


def dense_scores(A, E, d, fun):
    D = A.toarray()
    w = np.linalg.eigvalsh(D)
    out = []
    for (i, j), dh in zip(E, d):
        Dt = D.copy()
        if i != j:
            Dt[i - 1, j - 1] += dh
            Dt[j - 1, i - 1] += dh
        else:
            Dt[i - 1, i - 1] += dh
        out.append(_trace_formula(fun, np.linalg.eigvalsh(Dt), w))
    return np.array(out), float(np.max(np.abs(w)))


@pytest.mark.parametrize("name", ["grid_Austria", "grid_England", "grid_Mexico", "grid_Sweden"])
@pytest.mark.parametrize("fun", ["exp", "sinh", "cosh"])
def test_weighted_scores_match_dense_truth_on_power_grids(name, fun):
    A = load_graph(name).astype(float)
    E, d = mixed_candidates(A, seed=len(name))
    truth, nrm = dense_scores(A, E, d, fun)
    tol = 1e-10 * F[fun](nrm)
    x, its, _ = OW.trace_fun_update_edges_w(A, E, d, tol, None, fun)
    bad = np.abs(x - truth) > 10 * tol
    if fun == "sinh":
        # sinh is odd: while the Krylov space around (i, j) closes no odd walk through the changed entries, the projected
        # change is zero up to rounding and the reference's lag-2 rule (trace_fun_update.m:104-118) stops at step 3 on
        # it - the reference's stop, the same one tests/test_oracle_nodes.py meets.  Every miss is such a stop, and the
        # same candidates scored with the rule off (tol = 0, 30 steps) meet dense truth.
        assert np.all(its[bad] == 3) and np.all(np.abs(x[bad]) < 1e-3 * tol), (E[bad], x[bad], truth[bad])
        x2, _, _ = OW.trace_fun_update_edges_w(A, E[bad], d[bad], 0.0, 30, fun)
        assert np.all(np.abs(x2 - truth[bad]) <= 10 * tol)
    else:
        assert not bad.any(), (E[bad], x[bad], truth[bad], tol)


def test_zero_value_scores_exactly_zero():
    A = load_graph("grid_Sweden").astype(float)
    E, _ = mixed_candidates(A, seed=3, n_edges=4, n_missing=2, n_loops=2)
    x, its, _ = OW.trace_fun_update_edges_w(A, E, 0.0, 1e-8, None, "exp")
    assert np.all(x == 0.0)
    assert np.all(its == 3)                                  # the lag-2 rule on three equal values


def test_uniform_values_equal_the_reference_candidate_loop():
    A = load_graph("grid_England").astype(float)
    E, _ = mixed_candidates(A, seed=5, n_edges=6, n_missing=3, n_loops=0)
    x, its, lk = OW.trace_fun_update_edges_w(A, E, -0.5, 1e-8, None, "cosh")
    for h, (i, j) in enumerate(E):
        U = np.zeros((A.shape[0], 2))
        U[i - 1, 0] = U[j - 1, 1] = 1.0
        ref = O.trace_fun_update(A, U, -np.array([[0.0, 1.0], [1.0, 0.0]]) / 2.0, 1e-8, None, 0, "cosh")
        assert (x[h], its[h], lk[h]) == ref


@pytest.mark.parametrize("miobi,order", [("break", "mult"), ("make", "min")])
def test_weighted_greedy_on_a_01_graph_is_the_unweighted_greedy(miobi, order):
    A = load_graph("oregon_A0").astype(float)
    c = O.compute_centrality(A, "eig")
    nrm = float(np.max(np.abs(np.linalg.eigvalsh(A.toarray()))))
    tol = 1e-8 * np.exp(nrm)
    k, Q = 3, 15
    e1, r1, A1 = O.greedy_krylov(A, k, Q, c, order, tol, None, miobi=miobi)
    e2, r2, A2, applied = OW.greedy_krylov_weighted(A, k, Q, c, order, tol, None, "exp", miobi)
    assert np.array_equal(e1, e2)
    assert r1 == r2
    assert (A1 != A2).nnz == 0
    assert np.all(applied == (-1.0 if miobi == "break" else 1.0))


def test_weighted_greedy_applies_what_it_scored():
    A = load_graph("grid_Austria").astype(float)
    c = O.compute_centrality(A, "eig")
    tol = 1e-10 * np.exp(float(np.max(np.abs(np.linalg.eigvalsh(A.toarray())))))
    edges, rob, A_new, applied = OW.greedy_krylov_weighted(A, 3, 12, c, "mult", tol, None, "exp", "break")
    D0, D1 = A.toarray(), A_new.toarray()
    for (i, j), dh in zip(edges, applied):
        assert dh == -D0[i - 1, j - 1] and D1[i - 1, j - 1] == 0.0 and D1[j - 1, i - 1] == 0.0
    # the summed scores are the change of tr exp from A to A_new (each score is exact to the tolerance)
    total = _trace_formula("exp", np.linalg.eigvalsh(D1), np.linalg.eigvalsh(D0))
    assert abs(rob - total) <= 10 * 3 * tol
