"""The node-removal oracle (oracle.nodes.trace_fun_update_node, oracle.nodes.greedy_krylov_nodes) against dense truth:
tr f(Ã) - tr f(A) by eigvalsh, Ã = A with the off-diagonal entries of row and column v zeroed (a_vv kept)."""
import numpy as np
import pytest
import scipy.sparse as sp

from conftest import load_graph

import oracle as O
import oracle.nodes as ON
from oracle.updates import _trace_formula

F = {"exp": np.exp, "sinh": np.sinh, "cosh": np.cosh}


def with_self_loops(A, count=25, seed=7):
    """A plus `count` seeded diagonal entries (weights 0.5 .. 2)."""
    rng = np.random.default_rng(seed)
    n = A.shape[0]
    idx = rng.choice(n, count, replace=False)
    D = sp.csr_matrix((rng.uniform(0.5, 2.0, count), (idx, idx)), shape=(n, n))
    return (A.astype(float) + D).tocsr()


def graph(name):
    if name == "oregon_A0_loops":
        return with_self_loops(load_graph("oregon_A0"))
    return load_graph(name).astype(float)


def dense_node_scores(A, nodes, name):
    D = A.toarray()
    w = np.linalg.eigvalsh(D)
    out = []
    for v in nodes:
        Dt = D.copy()
        d = Dt[v - 1, v - 1]
        Dt[v - 1, :] = 0.0
        Dt[:, v - 1] = 0.0
        Dt[v - 1, v - 1] = d
        out.append(_trace_formula(name, np.linalg.eigvalsh(Dt), w))
    return np.array(out), float(np.max(np.abs(w)))


def top_nodes(A, count):
    c = O.compute_centrality(A, "eig")
    return np.argsort(-c, kind="stable")[:count] + 1


@pytest.mark.parametrize("name", ["oregon_A0", "transport_Anaheim", "grid_England", "oregon_A0_loops"])
@pytest.mark.parametrize("fun", ["exp", "sinh", "cosh"])
def test_node_score_matches_dense_truth_on_top_centrality_nodes(name, fun):
    A = graph(name)
    nodes = top_nodes(A, 40)
    truth, nrm = dense_node_scores(A, nodes, fun)
    tol = 1e-12 * F[fun](nrm)
    res = [ON.trace_fun_update_node(A, v, tol, None, fun) for v in nodes]
    x = np.array([r[0] for r in res])
    its = np.array([r[1] for r in res])
    bad = np.abs(x - truth) > 10 * tol
    if fun == "sinh":
        # The reference's lag-2 rule (trace_fun_update.m:104-118) compares step j with step j-2.  sinh is odd, and while
        # the Krylov space around v holds no odd cycle its projected change is zero up to rounding: the rule then stops
        # at step 3 on a value that has not moved yet.  On the road networks this hits a few of the top-40 nodes; every
        # such miss is a step-3 stop on a rounding-level value, every other node agrees.
        assert np.all(its[bad] == 3) and np.all(np.abs(x[bad]) < tol), (nodes[bad], x[bad], truth[bad])
        if name.startswith("oregon"):
            assert not bad.any()
    else:
        assert not bad.any(), (nodes[bad], x[bad], truth[bad], tol)
        assert np.all(its > 3)


def test_zero_degree_node_scores_zero_with_lucky_breakdown():
    A = sp.lil_matrix(load_graph("oregon_A0").astype(float))
    n = A.shape[0]
    v = 5
    for j in A.rows[v - 1][:]:
        A[v - 1, j] = 0.0
        A[j, v - 1] = 0.0
    A[v - 1, v - 1] = 1.5                                   # a self loop alone is no edge to remove
    A = A.tocsr()
    A.eliminate_zeros()
    for fun in ("exp", "sinh", "cosh"):
        assert ON.trace_fun_update_node(A, v, 1e-8, min(100, n), fun) == (0.0, 1, True)


def test_leaf_score_equals_the_removal_of_its_only_edge():
    A = load_graph("oregon_A0").astype(float)
    deg = np.diff(A.indptr)
    leaves = np.flatnonzero(deg == 1)[:5] + 1
    assert leaves.size == 5
    D = A.toarray()
    w = np.linalg.eigvalsh(D)
    nrm = float(np.max(np.abs(w)))
    for fun in ("exp", "cosh"):
        tol = 1e-12 * F[fun](nrm)
        for v in leaves:
            u = int(A.indices[A.indptr[v - 1]])
            U = np.zeros((A.shape[0], 2))
            U[v - 1, 0] = U[u, 1] = 1.0
            Dt = D + U @ np.array([[0.0, -1.0], [-1.0, 0.0]]) @ U.T
            edge = _trace_formula(fun, np.linalg.eigvalsh(Dt), w)
            x, _, _ = ON.trace_fun_update_node(A, v, tol, None, fun)
            assert abs(x - edge) <= 10 * tol, (v, x, edge)


def test_greedy_nodes_oracle_picks_the_exhaustive_dense_choice():
    A = load_graph("oregon_A0").astype(float)
    c = O.compute_centrality(A, "eig")
    nrm = float(np.max(np.abs(np.linalg.eigvalsh(A.toarray()))))
    tol = 1e-12 * np.exp(nrm)
    k, Q = 3, 25
    nodes, rob, A_new = ON.greedy_krylov_nodes(A, k, Q, c, tol, None, "exp")
    # exhaustive: the same candidate rule, every candidate scored densely
    top = list(np.argsort(-c, kind="stable")[:Q + k] + 1)
    B = A.copy()
    want, total = [], 0.0
    for _ in range(k):
        cand = top[:Q]
        vals, _ = dense_node_scores(B, cand, "exp")
        best = int(np.argmin(vals))
        v = cand[best]
        want.append(v)
        total += vals[best]
        B = B.tolil()
        for j in B.rows[v - 1][:]:
            if j != v - 1:
                B[v - 1, j] = 0.0
                B[j, v - 1] = 0.0
        B = B.tocsr()
        B.eliminate_zeros()
        top.remove(v)
    assert list(nodes) == want
    assert abs(rob - total) <= 10 * k * tol
    assert (A_new != B).nnz == 0
    for v in nodes:                                          # the chosen nodes are cut off
        row = A_new.getrow(v - 1)
        assert set(row.indices) <= {v - 1}


def test_greedy_nodes_oracle_rejects_unsymmetric():
    A = sp.csr_matrix(np.array([[0.0, 1.0], [0.0, 0.0]]))
    with pytest.raises(ValueError, match="GREEDY_KRYLOV:: Adjacency matrix should be symmetric"):
        ON.greedy_krylov_nodes(A, 1, 1, np.ones(2))
