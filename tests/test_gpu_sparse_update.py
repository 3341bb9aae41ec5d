"""tr f(Ã) - tr f(Ã - D) on the device (kr_trace_fun_sparse_update, csrc/sparse_update.cuh and the direction flavour of
csrc/entries_local.cuh) against the oracle (oracle.sparse_update, itself held to dense truth in
tests/test_oracle_sparse_update.py): 1e-10 relative with equal q; bit-identical repeats; the objective slice of the
reference's all-edges golden; the local path against the dense batch (KR_ENTRIES_LOCAL=0) at 1e-12 through every tier,
the step-limit fallback, a power-law graph, pattern-only and valued storage, edges that X removes and pending edits;
argument errors, fun_and_grad_all_edges(objective=True) and the MEX op."""
import json
import os
import sys
import warnings

import numpy as np
import pytest
import scipy.io as sio
import scipy.sparse as sp

from conftest import GOLDEN, ROOT, load_graph
from test_oracle_sparse_update import case, tol_for

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def kr():
    import krylov_robustness_b200 as kr
    return kr


def local_vs_dense(kr, monkeypatch, M, X, Om, fun, tol, it, qmax=32):
    loc = kr.trace_fun_sparse_update(M, X, Om, fun, tol, it, qmax, return_info=True)
    monkeypatch.setenv("KR_ENTRIES_LOCAL", "0")
    den = kr.trace_fun_sparse_update(M, X, Om, fun, tol, it, qmax, return_info=True)
    monkeypatch.delenv("KR_ENTRIES_LOCAL")
    assert loc[1] == den[1], (loc, den)
    assert abs(loc[0] - den[0]) <= 1e-12 * abs(den[0]), (loc[0], den[0])
    assert den[3]["tier_columns"] == [0, 0, 0]
    return loc


def road_case(name, m, seed=3):
    """A / max(A) of a road network, m random edges, X in [-0.5 a, 0.5 a]; returns Ã, X, Ω."""
    import oracle.sparse_update as S
    A = sp.csr_matrix(load_graph(name)).astype(np.float64)
    A = (A / A.max()).tocsr()
    rng = np.random.default_rng(seed)
    L = sp.tril(A, -1).tocoo()
    pick = rng.choice(L.nnz, m, replace=False)
    Om = np.stack([L.row[pick] + 1, L.col[pick] + 1], 1).astype(np.int64)
    X = (rng.random(m) - 0.5) * L.data[pick]
    return (A + S.delta(X, Om, A.shape[0])).tocsr(), X, Om


@pytest.mark.parametrize("name", ["transport_Anaheim", "grid_England", "grid_Mexico", "oregon_A0"])
@pytest.mark.parametrize("fun", ["exp", "sinh", "cosh"])
def test_device_matches_oracle(kr, name, fun):
    import oracle.sparse_update as S
    At, X, Om = case(name)
    tol = tol_for(At, fun)
    ref = S.trace_fun_sparse_update(At, X, Om, fun, tol, 100)
    M = kr.Matrix(At)
    dev = kr.trace_fun_sparse_update(M, X, Om, fun, tol, 100)
    assert dev[1] == ref[1], (dev, ref)
    assert abs(dev[0] - ref[0]) <= 1e-10 * abs(ref[0]), (dev, ref)
    again = kr.trace_fun_sparse_update(M, X, Om, fun, tol, 100)
    assert again == dev                                   # bit-identical, same q and iteration count


def test_zero_direction_and_removed_edges(kr):
    import oracle.sparse_update as S
    At, X, Om = case("transport_Anaheim")
    assert kr.trace_fun_sparse_update(At, 0 * X, Om, "sinh", 1e-10, 100) == (0.0, 0, 0)
    # X_h = -A(i, j): the edge is gone from Ã but present in A_t for t < 1
    A = sp.csr_matrix(load_graph("transport_Anaheim")).astype(np.float64)
    A = (A / A.max()).tocsr()
    L = sp.tril(A, -1).tocoo()
    Om2 = np.stack([L.row[:12] + 1, L.col[:12] + 1], 1).astype(np.int64)
    X2 = -L.data[:12].copy()
    X2[6:] *= 0.5
    At2 = (A + S.delta(X2, Om2, A.shape[0])).tocsr()
    At2.eliminate_zeros()
    assert At2.nnz == A.nnz - 12
    tol = tol_for(At2, "cosh")
    ref = S.trace_fun_sparse_update(At2, X2, Om2, "cosh", tol, 100)
    dev = kr.trace_fun_sparse_update(At2, X2, Om2, "cosh", tol, 100)
    assert dev[1] == ref[1] and abs(dev[0] - ref[0]) <= 1e-10 * abs(ref[0]), (dev, ref)


def test_reference_golden_objective(kr):
    """Anaheim, Ω = all 634 edges, f = sinh: the objective slice of the reference's literal call, at the tolerance the
    gradient of the sparse formulation is checked with (tests/test_reference_goldens.py)."""
    ref = json.load(open(os.path.join(GOLDEN, "reference_golden.json")))["Anaheim_all_edges_fg_sinh"]
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        I = sio.loadmat(os.path.join(GOLDEN, "reference_inputs.mat"))
    An = sp.csr_matrix(I["Anaheim"])
    OmA, XA = I["Anaheim_Omega"].astype(np.int64), I["Anaheim_X"].ravel()
    tol = 1e-10 * np.cosh(float(kr.normest(kr.Matrix(An), 1e-6)[0]))
    f, gr = kr.fun_and_grad_all_edges(XA, An, OmA, "sinh", "cosh", tol, 100, objective=True)
    assert abs(f - ref[0]) <= 1e-9 * abs(ref[0]), (f, ref[0])
    gr0 = kr.fun_and_grad_all_edges(XA, An, OmA, "sinh", "cosh", tol, 100)
    assert np.array_equal(gr, gr0)


def test_local_tiers_against_dense(kr, monkeypatch):
    # a tight tol on a road network: the spaces take more steps and outgrow the first budgets (at 1e-15 * cosh(||A||)
    # the lag-3 test compares rounding noise and the two paths may stop steps apart)
    At, X, Om = road_case("transport_Vermont", 3000)
    M = kr.Matrix(At)
    tol = 1e-12 * np.cosh(float(kr.normest(M, 1e-2)[0]))
    loc = local_vs_dense(kr, monkeypatch, M, X, Om, "sinh", tol, 100)
    tiers = loc[3]["tier_columns"]
    assert tiers[1] > 0 and tiers[2] > 0, loc


def test_step_limit_fallback_per_node(kr, monkeypatch):
    # tol = 0: every space runs to it = 30 > 24 steps, so every (start node, node) column takes the dense batch
    At, X, Om = road_case("transport_Anaheim", 40)
    loc = local_vs_dense(kr, monkeypatch, kr.Matrix(At), X, Om, "exp", 0.0, 30, qmax=3)
    R = np.unique(Om[:, 0]).size
    assert loc[1] == 3 and loc[2] == 30 and loc[3]["dense_columns"] == 3 * R


def test_power_law_graph_falls_back(kr, monkeypatch):
    At, X, Om = case("oregon_A7", m=60)
    M = kr.Matrix(At)
    loc = local_vs_dense(kr, monkeypatch, M, X, Om, "cosh", tol_for(At, "cosh"), 100)
    assert loc[3]["dense_columns"] > 0


@pytest.mark.parametrize("valued", [False, True])
def test_pattern_only_and_valued_storage(kr, monkeypatch, valued):
    import oracle.sparse_update as S
    A = sp.csr_matrix(load_graph("transport_Barcelona")).astype(np.float64)
    A.data[:] = 0.5
    rng = np.random.default_rng(5)
    L = sp.tril(A, -1).tocoo()
    pick = rng.choice(L.nnz, 200, replace=False)
    Om = np.stack([L.row[pick] + 1, L.col[pick] + 1], 1).astype(np.int64)
    X = 0.25 * rng.random(200)
    # pattern-only: Ã is the unweighted graph and the direction lowers the edges of Ω; valued: Ã = A + Δ
    At = (A + S.delta(X, Om, A.shape[0])).tocsr() if valued else A
    M = kr.Matrix(At)
    assert M.info()["pattern_only"] == (not valued)
    local_vs_dense(kr, monkeypatch, M, X, Om, "sinh", 1e-12 * np.cosh(float(kr.normest(M, 1e-2)[0])), 100)


def test_pending_edits(kr, monkeypatch):
    At, X, Om = road_case("transport_Anaheim", 60)
    B = At.tolil()
    i, j = int(Om[0, 0]), int(Om[0, 1])
    edits = [(i, j, 0.7), (3, 200, 0.4), (9, 9, 0.2)]
    M = kr.Matrix(At)
    for a, b, v in edits:
        M.set_edges([a], [b], v)
        B[a - 1, b - 1] = v
        B[b - 1, a - 1] = v
    B = B.tocsr()
    tol = 1e-12 * np.cosh(2.0)
    dev = kr.trace_fun_sparse_update(M, X, Om, "exp", tol, 100)
    ref = kr.trace_fun_sparse_update(B, X, Om, "exp", tol, 100)
    assert dev[1:] == ref[1:] and abs(dev[0] - ref[0]) <= 1e-12 * abs(ref[0]), (dev, ref)
    M2 = kr.Matrix(At)
    M2.set_edges([3], [200], 0.4)
    local_vs_dense(kr, monkeypatch, M2, X, Om, "exp", tol, 100)


def test_argument_errors(kr):
    At, X, Om = case("grid_England", m=10)
    n = At.shape[0]
    M = kr.Matrix(At)
    with pytest.raises(kr._lib.KrylovB200Error, match="Omega index out of range"):
        kr.trace_fun_sparse_update(M, [0.1], [[1, n + 1]], "exp", 1e-10, 50)
    with pytest.raises(kr._lib.KrylovB200Error, match="Omega index out of range"):
        kr.trace_fun_sparse_update(M, [0.1], [[0, 2]], "exp", 1e-10, 50)
    with pytest.raises(kr._lib.KrylovB200Error, match="qmax must be >= 1"):
        kr.trace_fun_sparse_update(M, X, Om, "exp", 1e-10, 50, qmax=0)
    with pytest.raises(ValueError, match="one value per row of Omega"):
        kr.trace_fun_sparse_update(M, X[:-1], Om, "exp", 1e-10, 50)
    with pytest.raises(ValueError, match="unsupported function"):
        kr.trace_fun_sparse_update(M, X, Om, "tanh", 1e-10, 50)
    U = sp.triu(At, format="csr")
    with pytest.raises(kr._lib.KrylovB200Error, match="FUN_AND_GRAD_KRYLOV_FCONNECTIVITY:: matrix A is not Hermitian"):
        kr.trace_fun_sparse_update(U, X, Om, "sinh", 1e-10, 50)
    with pytest.raises(kr._lib.KrylovB200Error, match="FUN_AND_GRAD_KRYLOV:: matrix A is not Hermitian"):
        kr.trace_fun_sparse_update(U, X, Om, "exp", 1e-10, 50)
    assert kr.trace_fun_sparse_update(M, [], np.zeros((0, 2)), "exp", 1e-10, 50) == (0.0, 0, 0)
    # qmax caps the order
    assert kr.trace_fun_sparse_update(M, X, Om, "exp", 0.0, 20, qmax=2)[1] == 2


def test_objective_option_of_fun_and_grad_all_edges(kr):
    import oracle.sparse_update as S
    A = sp.csr_matrix(load_graph("grid_Mexico")).astype(np.float64)
    A = (A / A.max()).tocsr()
    L = sp.tril(A, -1).tocoo()
    Om = np.vstack([np.stack([L.row + 1, L.col + 1], 1), [[4, 4]]]).astype(np.int64)
    X = 0.1 * np.random.default_rng(4).random(Om.shape[0])
    tol = 1e-10 * np.cosh(float(kr.normest(A, 1e-2)[0]))
    f, gr = kr.fun_and_grad_all_edges(X, A, Om, "sinh", "cosh", tol, 100, objective=True)
    assert np.array_equal(gr, kr.fun_and_grad_all_edges(X, A, Om, "sinh", "cosh", tol, 100))
    # Atilde = A + D + D' there: the diagonal pair enters twice
    D = sp.csr_matrix((X, (Om[:, 0] - 1, Om[:, 1] - 1)), shape=A.shape)
    At = (A + D + D.T).tocsr()
    Xd = np.where(Om[:, 0] == Om[:, 1], 2 * X, X)
    ref = S.trace_fun_sparse_update(At, Xd, Om, "sinh", tol, 100)[0]
    assert abs(f + ref) <= 1e-10 * abs(ref)


def test_mex_op_matches_python_binding(kr, tmp_path):
    sys.path.insert(0, os.path.join(ROOT, "tests", "mex_stub"))
    import bridge
    H = bridge.MexHost(bridge.build_host(tmp_path))
    At, X, Om = case("transport_Anaheim")
    tol = tol_for(At, "sinh")
    dtr, q, it = kr.trace_fun_sparse_update(At, X, Om, "sinh", tol, 100)
    out = H.call(["trace_fun_sparse_update", At, Om.astype(float), X[:, None], "sinh", tol, 100.0, 32.0], 3)
    assert out[0].ravel()[0] == dtr
    assert out[1].ravel()[0] == q and out[2].ravel()[0] == it
