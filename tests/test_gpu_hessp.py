"""Hessian times vectors on the device (kr_frechet_hessian_multiply, csrc/frechet.cuh) against the oracle (oracle.hessp,
itself held to dense truth in tests/test_oracle_hessp.py): 1e-10 relative to max |W| with equal iter in both forms,
bit-identical repeats; the reference form against the device's hessianfcn_fun and the Mexico goldens; the objective
form against a central difference of fun_and_grad_all_edges and against dense truth; pending edits, an edge that X
removes, argument errors, Y = 0, the MEX op and the MATLAB wrapper."""
import io
import json
import os
import sys
import warnings

import numpy as np
import pytest
import scipy.io as sio
import scipy.sparse as sp

from conftest import GOLDEN, ROOT, load_graph
from test_oracle_hessp import dense_truth

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def kr():
    import krylov_robustness_b200 as kr
    return kr


def case(name, m=24, seed=4):
    """A / max(A), m random edges with X in [-0.3, 0.3] a_ij, plus a non-edge, a diagonal pair, a duplicate and an edge
    that X removes completely (X = -a_ij)."""
    A = sp.csr_matrix(load_graph(name)).astype(np.float64)
    A = (A / A.max()).tocsr()
    n = A.shape[0]
    rng = np.random.default_rng(seed)
    L = sp.tril(A, -1).tocoo()
    pick = rng.choice(L.nnz, m + 1, replace=False)
    Om = np.stack([L.row[pick] + 1, L.col[pick] + 1], 1)
    X = (rng.random(m + 1) - 0.5) * 0.6 * L.data[pick]
    X[-1] = -L.data[pick[-1]]
    assert A[0, n - 1] == 0
    Om = np.vstack([Om, [[1, n], [5, 5], Om[0]]]).astype(np.int64)
    X = np.concatenate([X, [0.2, -0.1, 0.05]])
    return A, X, Om, rng


def tol_for(A, X, Om, fun):
    import oracle as O
    from test_oracle_hessp import atilde
    return 1e-10 * np.cosh(O.normest(sp.csr_matrix(atilde(A, X, Om)), 1e-2)[0])


@pytest.mark.parametrize("name", ["transport_Anaheim", "grid_England", "grid_Mexico", "oregon_A0"])
@pytest.mark.parametrize("fun", ["exp", "sinh", "cosh"])
def test_device_matches_oracle(kr, name, fun):
    import oracle.hessp as HP
    A, X, Om, rng = case(name)
    tol = tol_for(A, X, Om, fun)
    Y3 = rng.standard_normal((len(Om), 3))
    for ref_form in (False, True):
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            want, it_o = HP.hessian_multiply(X, A, Om, fun, Y3, tol, 64, reference_form=ref_form)
            got, it_d, info = kr.hessp_all_edges(X, A, Om, fun, Y3, tol, 64, reference_form=ref_form, return_info=True)
            again = kr.hessp_all_edges(X, A, Om, fun, Y3, tol, 64, reference_form=ref_form)
            one = kr.hessp_all_edges(X, A, Om, fun, Y3[:, 1], tol, 64, reference_form=ref_form)
        assert it_d == it_o
        assert np.abs(got - want).max() <= 1e-10 * np.abs(want).max(), (ref_form, np.abs(got - want).max())
        assert np.array_equal(got, again)
        assert one.shape == (len(Om),) and np.array_equal(one, got[:, 1])   # columns are independent: p = 1 is column r
        if name == "oregon_A0":           # power-law: balls outgrow every tier, those pairs take the dense families
            assert info["dense_pairs"] > 0, info
        else:
            assert info["tier_pairs"][0] == len(Om), info


def test_reference_form_equals_hessianfcn_and_the_goldens(kr):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        I = sio.loadmat(os.path.join(GOLDEN, "reference_inputs.mat"))
    ref = json.load(open(os.path.join(GOLDEN, "reference_golden.json")))
    A, Om, X = sp.csr_matrix(I["Mexico"]), I["Mexico_Omega"].astype(np.int64), I["Mexico_X"].ravel()
    m = len(Om)
    Y = np.random.default_rng(5).standard_normal((m, 3))
    for fun, key in (("exp", "Mexico_hessian_exp"), ("sinh", "Mexico_hessian_sinh")):
        W = kr.hessp_all_edges(X, A, Om, fun, Y, 1e-10, 100, reference_form=True)
        for Hes in (kr.hessianfcn_fun(X, A, Om, fun, 1e-10, 100),
                    np.asarray(ref[key], dtype=np.float64).reshape(m, m, order="F")):
            HY = Hes @ Y
            assert np.abs(W - HY).max() <= 1e-10 * np.abs(HY).max(), key


def test_objective_form_is_the_hessian_of_the_gradient(kr):
    """Anaheim: the product against a central difference of fun_and_grad_all_edges (sinh objective, cosh gradient, so
    the derivative taken is that of cosh) and against dense truth."""
    A = sp.csr_matrix(load_graph("transport_Anaheim")).astype(np.float64)
    A = (A / A.max()).tocsr()
    rng = np.random.default_rng(6)
    L = sp.tril(A, -1).tocoo()
    pick = rng.choice(L.nnz, 30, replace=False)
    Om = np.stack([L.row[pick] + 1, L.col[pick] + 1], 1).astype(np.int64)
    X = (rng.random(30) - 0.5) * 0.4 * L.data[pick]
    y = rng.standard_normal(30)
    tol = 1e-12
    W = kr.hessp_all_edges(X, A, Om, "cosh", y, tol, 64)
    eps = 1e-4
    gp = kr.fun_and_grad_all_edges(X + eps * y, A, Om, "sinh", "cosh", tol, 64)
    gm = kr.fun_and_grad_all_edges(X - eps * y, A, Om, "sinh", "cosh", tol, 64)
    fd = (gp - gm) / (2 * eps)
    assert np.abs(W - fd).max() <= 1e-6 * np.abs(fd).max()
    T = dense_truth(A, X, Om, "cosh", y[:, None], False)[:, 0]
    assert np.abs(W - T).max() <= 1e-9 * np.abs(T).max()


def test_pending_edits_and_resident_matrix(kr):
    """A resident Matrix of Atilde with pending set_edges edits gives what the edited matrix gives."""
    A, X, Om, rng = case("transport_Anaheim", m=16)
    from test_oracle_hessp import atilde
    At = sp.csr_matrix(atilde(A, X, Om))
    M = kr.Matrix(At)
    i, j = np.array([Om[2, 0], Om[3, 0], 7]), np.array([Om[2, 1], 9, 7])
    M.set_edges(i, j, np.array([0.0, 0.3, 0.4]))
    E = At.tolil()
    for a, b, v in zip(i, j, [0.0, 0.3, 0.4]):
        E[a - 1, b - 1] = v
        E[b - 1, a - 1] = v
    E = E.tocsr()
    E.eliminate_zeros()
    Y = rng.standard_normal((len(Om), 2))
    tol = 1e-11
    got = kr.hessp_all_edges(None, M, Om, "sinh", Y, tol, 64)
    want = kr.hessp_all_edges(np.zeros(len(Om)), E, Om, "sinh", Y, tol, 64)
    assert np.abs(got - want).max() <= 1e-12 * np.abs(want).max()


def test_argument_errors_and_zero_y(kr):
    A, X, Om, rng = case("transport_Anaheim", m=8)
    n = A.shape[0]
    Y = rng.standard_normal(len(Om))
    assert np.array_equal(kr.hessp_all_edges(X, A, Om, "exp", 0 * Y, 1e-10, 64), np.zeros(len(Om)))
    assert kr.hessp_all_edges(X, A, Om, "exp", np.zeros((len(Om), 0)), 1e-10, 64).shape == (len(Om), 0)
    with pytest.raises(Exception, match="out of range"):
        kr.hessp_all_edges(None, kr.Matrix(A), np.vstack([Om, [[1, n + 1]]]), "exp", np.append(Y, 1.0), 1e-10, 64)
    with pytest.raises(Exception, match="it must be"):
        kr.hessp_all_edges(X, A, Om, "exp", Y, 1e-10, 0)
    with pytest.raises(ValueError, match="one row per row"):
        kr.hessp_all_edges(X, A, Om, "exp", Y[:-1], 1e-10, 64)
    U = sp.csr_matrix(A).tolil()
    U[0, 1] = 5.0
    M = kr.Matrix(U.tocsr())
    with pytest.raises(Exception, match="FUN_AND_GRAD_KRYLOV:: matrix A is not Hermitian"):
        kr.hessp_all_edges(None, M, Om, "exp", Y, 1e-10, 64)
    with pytest.raises(Exception, match="FCONNECTIVITY:: matrix A is not Hermitian"):
        kr.hessp_all_edges(None, M, Om, "cosh", Y, 1e-10, 64)
    # p < 0 through the C ABI
    from krylov_robustness_b200.engine import _ptr
    Mt = kr.Matrix(sp.csr_matrix(A))
    Omf = np.asfortranarray(Om)
    W = np.zeros(len(Om))
    st = Mt.ctx.lib.kr_frechet_hessian_multiply(Mt.ctx.h, Mt.h, len(Om), _ptr(Omf), -1, _ptr(Y), len(Om), 0, 0, 1e-10,
                                                64, _ptr(W), len(Om), None, None)
    assert st != 0 and "p must be" in Mt.ctx.lib.kr_last_error().decode()


def test_mex_op_and_matlab_wrapper(kr, tmp_path):
    sys.path.insert(0, os.path.join(ROOT, "tests", "mex_stub"))
    import bridge
    from oracle.mlab import Interpreter
    H = bridge.MexHost(bridge.build_host(tmp_path))
    A, X, Om, rng = case("transport_Anaheim", m=12)
    from test_oracle_hessp import atilde
    At = sp.csr_matrix(atilde(A, X, Om))
    Y = rng.standard_normal((len(Om), 2))
    tol = 1e-10
    want, it = kr.hessp_all_edges(X, A, Om, "cosh", Y, tol, 64, return_info=True)[:2]
    out = H.call(["hessian_multiply", At, Om.astype(float), Y, "cosh", tol, 64.0, 0.0], 2)
    assert np.array_equal(out[0].reshape(Y.shape, order="F"), want) and out[1].ravel()[0] == it
    ref = kr.hessp_all_edges(X, A, Om, "cosh", Y, tol, 64, reference_form=True)
    out = H.call(["hessian_multiply", At, Om.astype(float), Y, "cosh", tol, 64.0, 1.0], 1)
    assert np.array_equal(out[0].reshape(Y.shape, order="F"), ref)
    # the wrapper as an fmincon HessianMultiplyFcn: a one-line closure over X
    I = Interpreter(stdout=io.StringIO())
    H.install(I)
    I.addpath(os.path.join(ROOT, "krylov_robustness_b200", "matlab"))
    script = tmp_path / "hmf.m"
    script.write_text("hmf = @(x, y) hessp_all_edges(x, A, Omega, @cosh, y, tol, 64);\nW = hmf(X, Y);\n")
    ws = I.run_script(str(script), {"A": sp.csc_matrix(A), "Omega": Om.astype(float), "tol": tol, "X": X[:, None],
                                    "Y": Y})
    assert np.abs(np.asarray(ws["W"]).reshape(Y.shape, order="F") - want).max() <= 1e-13 * np.abs(want).max()


def local_vs_dense(kr, monkeypatch, M, Om, fun, Y, tol, it, reference_form=False):
    loc = kr.hessp_all_edges(None, M, Om, fun, Y, tol, it, reference_form=reference_form, return_info=True)
    monkeypatch.setenv("KR_ENTRIES_LOCAL", "0")
    den = kr.hessp_all_edges(None, M, Om, fun, Y, tol, it, reference_form=reference_form, return_info=True)
    monkeypatch.delenv("KR_ENTRIES_LOCAL")
    assert loc[1] == den[1], (loc[1:], den[1:])
    assert np.abs(loc[0] - den[0]).max() <= 1e-12 * np.abs(den[0]).max()
    assert den[2] == {"tier_pairs": [0, 0, 0], "dense_pairs": len(Om)}
    return loc


def vermont(m=None, seed=4):
    A = sp.csr_matrix(load_graph("transport_Vermont")).astype(np.float64)
    A = (A / A.max()).tocsr()
    L = sp.tril(A, -1).tocoo()
    Om = np.stack([L.row + 1, L.col + 1], 1).astype(np.int64)
    X = 0.1 * L.data * np.random.default_rng(seed).random(L.nnz)
    n = A.shape[0]
    D = sp.csr_matrix((X, (Om[:, 0] - 1, Om[:, 1] - 1)), shape=(n, n))
    return A, X, Om, (A + D + D.T).tocsr()


def test_local_vs_dense_through_the_tiers(kr, monkeypatch):
    """A tight tol on 2 000 Vermont edges: the balls of the longer pairs outgrow the first tier."""
    import oracle as O
    A, X, Om, At = vermont()
    rng = np.random.default_rng(7)
    Om = Om[rng.choice(len(Om), 2000, replace=False)]
    tol = 1e-13 * np.cosh(O.normest(At, 1e-2)[0])
    M = kr.Matrix(At)
    loc = local_vs_dense(kr, monkeypatch, M, Om, "cosh", rng.standard_normal((len(Om), 2)), tol, 24)
    assert loc[2]["tier_pairs"][1] > 0, loc[2]


def test_local_vs_dense_step_limit_pattern_valued_pending(kr, monkeypatch):
    A, X, Om, rng = case("transport_Anaheim", m=20)
    from test_oracle_hessp import atilde
    At = sp.csr_matrix(atilde(A, X, Om))
    Y = rng.standard_normal((len(Om), 3))
    # step limit: tol = 0 never stops, it > 24 is beyond the local path: every pair takes the dense families
    loc = local_vs_dense(kr, monkeypatch, kr.Matrix(At), Om, "sinh", Y, 0.0, 30)
    assert loc[1] == 30 and loc[2]["dense_pairs"] == len(Om)
    # valued storage, both forms
    for ref_form in (False, True):
        loc = local_vs_dense(kr, monkeypatch, kr.Matrix(At), Om, "exp", Y, 1e-10, 64, ref_form)
        assert loc[2]["dense_pairs"] == 0
    # pattern-only storage (every stored value 0.25, X = 0)
    P = sp.csr_matrix(load_graph("transport_Anaheim"))
    P.data[:] = 0.25
    Mp = kr.Matrix(P)
    loc = local_vs_dense(kr, monkeypatch, Mp, Om, "cosh", Y, 1e-10, 64)
    assert loc[2]["dense_pairs"] == 0
    # pending edits, folded in before either path runs
    Me = kr.Matrix(At)
    Me.set_edges(np.array([Om[2, 0], Om[3, 0]]), np.array([Om[2, 1], 9]), np.array([0.0, 0.3]))
    local_vs_dense(kr, monkeypatch, Me, Om, "sinh", Y, 1e-10, 64)


def test_vermont_all_edges(kr):
    """All 104 644 edges on the local path; 20 sampled rows against the oracle's rows= evaluation."""
    import oracle as O
    import oracle.hessp as HP
    A, X, Om, At = vermont()
    tol = 1e-8 * np.cosh(O.normest(At, 1e-2)[0])
    rng = np.random.default_rng(8)
    Y = rng.standard_normal((len(Om), 2))
    W, it, info = kr.hessp_all_edges(None, kr.Matrix(At), Om, "cosh", Y, tol, 100, return_info=True)
    assert info["dense_pairs"] == 0 and info["tier_pairs"][0] == len(Om), info
    rows = rng.choice(len(Om), 20, replace=False)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        want, _ = HP.hessian_multiply(X, A, Om, "cosh", Y, tol, 100, rows=rows)
    assert np.abs(W[rows] - want).max() <= 1e-10 * np.abs(want).max()
