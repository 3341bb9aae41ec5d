"""Node-removal scores on the device (kr_trace_fun_update_nodes, csrc/nodes.cuh) against the oracle
(oracle.nodes.trace_fun_update_node, itself held to dense truth in tests/test_oracle_nodes.py): values to 1e-10 relative,
iteration counts and lucky flags equal; bit-reproducible; pending edge edits; replicas; the greedy node driver; the
MEX op."""
import os
import sys

import numpy as np
import pytest
import scipy.sparse as sp

from conftest import ROOT, load_graph

pytestmark = pytest.mark.gpu

F = {"exp": np.exp, "sinh": np.sinh, "cosh": np.cosh}


@pytest.fixture(scope="module")
def kr():
    import krylov_robustness_b200 as kr
    return kr


_GRAPHS = {}


def graph(name):
    if name not in _GRAPHS:
        if name == "powerlaw_50k":
            # above the L2-resident cut (CSR_L2_RESIDENT_NNZ = 400 000 stored entries)
            from krylov_robustness_b200.graphs import power_law_graph
            A = power_law_graph(50_000, 600_000, 2.2, 11)
        else:
            A = load_graph(name)
        _GRAPHS[name] = sp.csr_matrix(A).astype(np.float64)
    return _GRAPHS[name]


def top_nodes(A, count):
    import oracle as O
    c = O.compute_centrality(A, "eig")
    return np.argsort(-c, kind="stable")[:count] + 1


def tol_for(A, fun):
    # 1e-8 * f(||A||): at 1e-12 * f(||A||) the lag-2 test on Oregon A7 compares differences at rounding level (scores
    # of hubs agree to ~6e-12 relative between two correct implementations), and the step at which it fires can differ
    # by one; the oracle's agreement with dense truth at 1e-12 is tests/test_oracle_nodes.py
    import oracle as O
    nrm, _ = O.normest(A, 1e-2)
    return 1e-8 * F[fun](nrm)


def oracle_scores(A, nodes, tol, it, fun):
    import oracle.nodes as ON
    res = [ON.trace_fun_update_node(A, int(v), tol, it, fun) for v in nodes]
    return (np.array([r[0] for r in res]), np.array([r[1] for r in res]), np.array([r[2] for r in res]))


def assert_matches(dev, ref, tol):
    x, it, lk = dev
    xo, ito, lko = ref
    assert np.array_equal(it, ito), (it, ito)
    assert np.array_equal(lk, lko)
    # 1e-10 relative; scores at rounding level (sinh on a node whose neighbourhood has no odd cycle yet, stopped by the
    # lag-2 rule at step 3) are compared against a floor far below tol
    err = np.abs(x - xo)
    assert np.all(err <= 1e-10 * np.abs(xo) + 1e-4 * tol), (err / np.maximum(np.abs(xo), 1e-300)).max()


@pytest.mark.parametrize("name", ["oregon_A0", "oregon_A7", "transport_Anaheim", "grid_England", "powerlaw_50k"])
@pytest.mark.parametrize("fun", ["exp", "sinh", "cosh"])
def test_device_matches_oracle(kr, name, fun):
    A = graph(name)
    nodes = top_nodes(A, 24)
    tol = tol_for(A, fun)
    M = kr.Matrix(A)
    it = min(100, A.shape[0])
    dev = kr.trace_fun_update_nodes(M, nodes, tol, it, fun)
    assert_matches(dev, oracle_scores(A, nodes, tol, it, fun), tol)
    assert np.all(dev[1] >= 3)


@pytest.mark.parametrize("it", [1, 2, 5, 9, 70])
def test_iteration_caps_that_are_hit(kr, it):
    # tol = 0: only the cap or a lucky breakdown stops a column; 9 ends one step past the first batch of 8, 70 > 64
    A = graph("transport_Anaheim")
    nodes = top_nodes(A, 20)
    dev = kr.trace_fun_update_nodes(A, nodes, 0.0, it, "exp")
    assert np.all(dev[1] == it)
    assert_matches(dev, oracle_scores(A, nodes, 0.0, it, "exp"), 1e-12)


def test_zero_degree_and_leaf_nodes(kr):
    A = sp.lil_matrix(graph("oregon_A0"))
    v = 7
    for j in A.rows[v - 1][:]:
        A[v - 1, j] = 0.0
        A[j, v - 1] = 0.0
    A = A.tocsr()
    A.eliminate_zeros()
    leaves = np.flatnonzero(np.diff(A.indptr) == 1)[:6] + 1
    nodes = np.concatenate([[v], leaves, [v]])
    tol = tol_for(A, "cosh")
    x, it, lk = kr.trace_fun_update_nodes(A, nodes, tol, None, "cosh")
    assert x[0] == 0.0 and it[0] == 1 and lk[0] and x[-1] == 0.0 and it[-1] == 1
    assert np.all(np.isfinite(x))
    assert_matches((x, it, lk), oracle_scores(A, nodes, tol, min(100, A.shape[0]), "cosh"), tol)


def test_bit_identical_on_repeat(kr):
    A = graph("powerlaw_50k")
    nodes = top_nodes(A, 40)
    M = kr.Matrix(A)
    tol = tol_for(A, "exp")
    a = kr.trace_fun_update_nodes(M, nodes, tol, 100, "exp")
    b = kr.trace_fun_update_nodes(M, nodes, tol, 100, "exp")
    for u, w in zip(a, b):
        assert np.array_equal(u, w)


def test_pending_edits_on_the_node_row_and_its_neighbours(kr):
    A = graph("oregon_A7")
    nodes = top_nodes(A, 12)
    v = int(nodes[0])
    nb = [int(j) + 1 for j in A.indices[A.indptr[v - 1]:A.indptr[v]] if j != v - 1]
    u = max(nb, key=lambda j: A.indptr[j] - A.indptr[j - 1])             # the neighbour with the most neighbours
    w = [int(j) + 1 for j in A.indices[A.indptr[u - 1]:A.indptr[u]] if j + 1 not in (u, v)][0]
    far = int(np.flatnonzero(np.diff(A.indptr) == 1)[0]) + 1
    edits = [(v, nb[1], 0.0),             # v's row: delete
             (v, far, 1.0),               # v's row: insert
             (v, nb[2], 0.5),             # v's row: change
             (v, v, 2.0),                 # v's own diagonal entry
             (u, w, 0.0),                 # a neighbour's row: delete
             (u, far, 1.5)]               # a neighbour's row: insert
    M = kr.Matrix(A)
    B = A.tolil()
    for i, j, val in edits:
        M.set_edges([i], [j], val)
        B[i - 1, j - 1] = val
        B[j - 1, i - 1] = val
    B = B.tocsr()
    B.eliminate_zeros()
    cand = np.concatenate([nodes, [u, w, far]])
    tol = tol_for(B, "exp")
    dev = kr.trace_fun_update_nodes(M, cand, tol, 100, "exp")
    assert_matches(dev, oracle_scores(B, cand, tol, 100, "exp"), tol)


def test_replicated_matrix_gives_identical_scores(kr):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("one GPU")
    A = graph("oregon_A7")
    nodes = top_nodes(A, 64)
    tol = tol_for(A, "exp")
    single = kr.trace_fun_update_nodes(kr.Matrix(A), nodes, tol, 100, "exp")
    multi = kr.Matrix(A)
    assert multi.replicate() >= 2
    shared = kr.trace_fun_update_nodes(multi, nodes, tol, 100, "exp")
    for u, w in zip(single, shared):
        assert np.array_equal(u, w)


def test_argument_errors(kr):
    A = graph("oregon_A0")
    n = A.shape[0]
    M = kr.Matrix(A)
    with pytest.raises(kr._lib.KrylovB200Error, match="node index out of range"):
        kr.trace_fun_update_nodes(M, [1, n + 1], 1e-8, 20)
    with pytest.raises(kr._lib.KrylovB200Error, match="node index out of range"):
        kr.trace_fun_update_nodes(M, [0], 1e-8, 20)
    with pytest.raises(kr._lib.KrylovB200Error, match="it must be in"):
        kr.trace_fun_update_nodes(M, [1], 1e-8, 0)
    with pytest.raises(kr._lib.KrylovB200Error, match="it must be in"):
        kr.trace_fun_update_nodes(M, [1], 1e-8, 129)
    with pytest.raises(ValueError, match="unsupported function"):
        kr.trace_fun_update_nodes(M, [1], 1e-8, 20, "tanh")
    U = sp.triu(A, format="csr")
    with pytest.raises(kr._lib.KrylovB200Error, match="KRYLOV_MIOBI:: Adjacency matrix should be symmetric"):
        kr.trace_fun_update_nodes(U, [1], 1e-8, 20)
    with pytest.raises(ValueError, match="GREEDY_KRYLOV:: Adjacency matrix should be symmetric"):
        kr.greedy_krylov_nodes(U, 1, 5, np.ones(n))
    x, it, lk = kr.trace_fun_update_nodes(M, [], 1e-8, 20)
    assert x.size == it.size == lk.size == 0


@pytest.mark.parametrize("name,fun", [("oregon_A0", "exp"), ("grid_England", "cosh")])
def test_greedy_nodes_device_matches_oracle(kr, name, fun):
    import oracle as O
    import oracle.nodes as ON
    A = graph(name)
    c = O.compute_centrality(A, "eig")
    tol = tol_for(A, fun)
    k, Q = 4, 20
    nd, rd, Ad = kr.greedy_krylov_nodes(A, k, Q, c, tol, None, fun)
    no, ro, Ao = ON.greedy_krylov_nodes(A, k, Q, c, tol, None, fun)
    assert list(nd) == list(no)
    assert abs(rd - ro) <= 1e-10 * abs(ro)
    assert (Ad != Ao).nnz == 0


def test_mex_op_matches_python_binding(kr, tmp_path):
    sys.path.insert(0, os.path.join(ROOT, "tests", "mex_stub"))
    import bridge
    H = bridge.MexHost(bridge.build_host(tmp_path))
    A = graph("oregon_A0")
    nodes = top_nodes(A, 30)
    tol = tol_for(A, "exp")
    x, it, lk = kr.trace_fun_update_nodes(A, nodes, tol, 100, "exp")
    out = H.call(["trace_fun_update_nodes", A, nodes.astype(float)[:, None], tol, 100.0, "exp"], 3)
    assert np.array_equal(out[0].ravel(), x)
    assert np.array_equal(out[1].ravel(), it.astype(float))
    assert np.array_equal(out[2].ravel(), lk.astype(float))
