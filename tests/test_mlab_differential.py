"""Differential test of the oracle against the reference's OWN sources on randomised inputs.

Only where a checkout of the reference is named by KR_REFERENCE_DIR: every case draws a small random graph and random
arguments, runs the reference's unmodified functions/*.m through the interpreter of oracle/mlab and the NumPy/SciPy
oracle on the same inputs, and requires the same values (1e-10), iteration counts, flags, warnings-relevant outcomes
and selected edges.  The committed golden files pin a fixed set of calls; this sweeps the argument space around them
(weighted graphs, self loops, rank-one and rank-four updates, unsymmetric omega lists, ties in the centrality,
iteration caps that are hit, shifted / unshifted expmv, both trace estimators)."""
import io
import os
import warnings

import numpy as np
import pytest
import scipy.sparse as sp

from oracle.mlab import Interpreter, FH

REFDIR = os.environ.get("KR_REFERENCE_DIR", "")
pytestmark = pytest.mark.skipif(not (REFDIR and os.path.isdir(os.path.join(REFDIR, "functions"))),
                                reason="KR_REFERENCE_DIR names no checkout of the reference: the committed goldens stand in")
RTOL = 1e-10


@pytest.fixture(scope="module")
def I():
    return Interpreter(path=[os.path.join(REFDIR, "functions")], stdout=io.StringIO())


@pytest.fixture(scope="module")
def O():
    import oracle
    return oracle


def graph(rng, n, deg=4.0, weighted=False, loops=0):
    """Connected-ish symmetric graph: a ring plus random chords."""
    m = int(n * deg / 2)
    i = np.concatenate([np.arange(n), rng.integers(0, n, m)])
    j = np.concatenate([(np.arange(n) + 1) % n, rng.integers(0, n, m)])
    keep = i != j
    A = sp.coo_matrix((np.ones(keep.sum()), (i[keep], j[keep])), shape=(n, n)).tocsr()
    A = ((A + A.T) > 0).astype(np.float64)
    if weighted:
        W = sp.triu(A, 1).tocoo()
        w = rng.uniform(0.2, 1.0, W.nnz)
        A = sp.coo_matrix((w, (W.row, W.col)), shape=(n, n)).tocsr()
        A = A + A.T
    if loops:
        d = rng.choice(n, loops, replace=False)
        A = A + sp.coo_matrix((np.ones(loops), (d, d)), shape=(n, n)).tocsr()
    A = sp.csr_matrix(A)
    A.sort_indices()
    return A


def close(a, b, rtol=RTOL):
    a = np.asarray(a)
    if np.iscomplexobj(a):                                   # MATLAB keeps a complex result whose imaginary parts cancelled
        assert np.max(np.abs(a.imag)) <= 1e-9 * max(np.max(np.abs(a.real)), 1e-300)
        a = a.real
    a, b = np.asarray(a, dtype=np.float64).ravel(order="F"), np.asarray(b, dtype=np.float64).ravel(order="F")
    assert a.shape == b.shape, (a.shape, b.shape)
    scale = max(np.max(np.abs(b)), 1e-300) if b.size else 1.0
    assert np.max(np.abs(a - b)) <= rtol * scale if b.size else True, (np.max(np.abs(a - b)) / scale)


def sc(v):
    return float(np.asarray(v).ravel()[0])


@pytest.mark.parametrize("seed", range(8))
def test_trace_fun_update_random(I, O, seed):
    rng = np.random.default_rng(100 + seed)
    n = int(rng.integers(140, 260))
    A = graph(rng, n, weighted=seed % 3 == 1, loops=3 if seed % 4 == 2 else 0)
    rk = int(rng.choice([1, 2, 2, 3, 4]))
    nodes = rng.choice(n, rk, replace=False)
    U = np.zeros((n, rk))
    U[nodes, np.arange(rk)] = 1.0
    B = rng.standard_normal((rk, rk))
    B = (B + B.T) / 2 if seed % 5 else np.triu(B)          # a non-Hermitian B every fifth case (no symmetrisation branch)
    fun = ["exp", "sinh", "cosh"][seed % 3]
    it = int(rng.choice([3, 6, 100]))                       # small caps are hit: "Reached maximum number of iterations"
    tol = 10.0 ** rng.integers(-12, -4)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        ox, oit, olk = O.trace_fun_update(A, U, B, tol, it, 0, fun)
    x, itr, lk = I.call("trace_fun_update", sp.csc_matrix(A), U, B, tol, it, 0, FH(fun), nargout=3)
    assert sc(itr) == oit and bool(sc(lk)) == bool(olk)
    close(x, ox)


@pytest.mark.parametrize("seed", range(5))
def test_fun_update_and_callbacks_random(I, O, seed):
    rng = np.random.default_rng(200 + seed)
    n = int(rng.integers(300, 420))
    A = graph(rng, n, weighted=True)
    T = sp.tril(A, -1).tocoo()
    pick = np.sort(rng.choice(T.nnz, int(rng.integers(2, 7)), replace=False))
    Om = np.stack([T.row[pick] + 1, T.col[pick] + 1], 1).astype(np.float64)
    X = 0.1 * rng.uniform(0, 1, len(pick)).reshape(-1, 1)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        nrm = O.normest(A, 1e-6)[0]
        eA, itE = O.function_multiple_entries(A, Om.astype(np.int64), "exp", 1e-10 * np.exp(nrm), 100)
        of, ogr = O.fun_and_grad_krylov_exp(X.ravel(), A, Om.astype(np.int64), eA, 1e-9, 100, 0)
        dfA, _ = O.function_multiple_entries(A, Om.astype(np.int64), "cosh", 1e-10 * np.cosh(nrm), 100)
        of2, ogr2 = O.fun_and_grad_krylov_fun(X.ravel(), A, Om.astype(np.int64), "sinh", "cosh", dfA, 1e-9, 100, 0)
        oH = O.hessianfcn_exp(X.ravel(), A, Om.astype(np.int64), 1e-9, 100)
        oH2 = O.hessianfcn_fun(X.ravel(), A, Om.astype(np.int64), "cosh", 1e-9, 100)
    Ac = sp.csc_matrix(A)
    reA, ritE = I.call("function_multiple_entries", Ac, Om, FH("exp"), 1e-10 * np.exp(nrm), 100, np.inf, 0, nargout=2)
    assert sc(ritE) == itE
    close(reA, eA)
    f, gr = I.call("fun_and_grad_krylov_exp", X, Ac, Om, np.asarray(eA).reshape(-1, 1), 1e-9, 100, 0, nargout=2)
    close(np.concatenate([[sc(f)], gr.ravel()]), np.concatenate([[of], np.ravel(ogr)]))
    rdfA = I.call("function_multiple_entries", Ac, Om, FH("cosh"), 1e-10 * np.cosh(nrm), 100, np.inf, 0, nargout=1)[0]
    close(rdfA, dfA)
    f2, gr2 = I.call("fun_and_grad_krylov_fun", X, Ac, Om, FH("sinh"), FH("cosh"), np.asarray(dfA).reshape(-1, 1), 1e-9, 100, 0,
                     nargout=2)
    close(np.concatenate([[sc(f2)], gr2.ravel()]), np.concatenate([[of2], np.ravel(ogr2)]))
    close(I.call("hessianfcn_exp", X, Ac, Om, 1e-9, 100, nargout=1)[0], oH)
    close(I.call("hessianfcn_fun", X, Ac, Om, FH("cosh"), 1e-9, 100, nargout=1)[0], oH2)


@pytest.mark.parametrize("seed", range(6))
def test_entries_with_repeated_rows_and_diagonal(I, O, seed):
    rng = np.random.default_rng(300 + seed)
    n = int(rng.integers(150, 300))
    A = graph(rng, n, weighted=seed % 2 == 0)
    k = int(rng.integers(3, 12))
    rows = rng.integers(1, n + 1, k)
    rows[k // 2:] = rows[: k - k // 2]                       # repeated first indices share one Krylov space
    cols = rng.integers(1, n + 1, k)
    cols[0] = rows[0]                                        # a diagonal entry
    Om = np.stack([rows, cols], 1).astype(np.float64)
    fun = ["exp", "cosh", "sinh"][seed % 3]
    it = 100 if seed % 3 else 5
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        oX, oit = O.function_multiple_entries(A, Om.astype(np.int64), fun, 1e-9, it)
    X, itr = I.call("function_multiple_entries", sp.csc_matrix(A), Om, FH(fun), 1e-9, it, np.inf, 0, nargout=2)
    assert sc(itr) == oit
    close(X, oX)


@pytest.mark.parametrize("seed", range(6))
def test_expmv_family_random(I, O, seed):
    rng = np.random.default_rng(400 + seed)
    n = int(rng.integers(120, 400))
    A = graph(rng, n, deg=6.0, weighted=seed % 2 == 1, loops=5 if seed % 3 == 0 else 0)
    q = int(rng.integers(1, 6))
    b = rng.standard_normal((n, q))
    t = float(rng.choice([1.0, 0.3, 2.5, -1.0]))
    shift = bool(seed % 2 == 0)
    full_term = bool(seed % 3 == 1)
    of, os_, om, omv, omvd, ounA = O.expmv(t, A, b, None, "double", shift, False, full_term)
    f, s, m, mv, mvd, unA = I.call("expmv", t, sp.csc_matrix(A), b, np.zeros((0, 0)), "double", shift, False, full_term, nargout=6)
    assert [sc(s), sc(m), sc(mv), sc(mvd), sc(unA)] == [os_, om, omv, omvd, ounA]
    close(f, of)
    oM, omv2, oal, ounA2 = O.select_taylor_degree(A, b, 55, 8, "double", shift, False, seed % 2 == 1)
    M, mv2, al, unA2 = I.call("select_taylor_degree", sp.csc_matrix(A), b, 55, 8, "double", shift, False, seed % 2 == 1, nargout=4)
    assert sc(mv2) == omv2 and sc(unA2) == ounA2
    close(al, oal, 1e-12)
    close(M, oM, 1e-12)
    p = int(rng.integers(2, 8))
    mu = A.diagonal().sum() / n
    for Bm in (A, (A - mu * sp.identity(n)).tocsr()):         # the non-negative branch and the normest1 branch
        oc, omvn = O.normAm(Bm, p)
        c, mvn = I.call("normAm", sp.csc_matrix(Bm), p, nargout=2)
        assert sc(mvn) == omvn
        close(c, oc, 1e-12)


@pytest.mark.parametrize("seed", range(4))
def test_mc_trace_and_trace_exp_random(I, O, seed, tmp_path):
    rng = np.random.default_rng(500 + seed)
    n = int(rng.integers(150, 300))
    A = graph(rng, n, weighted=seed % 2 == 0) * 0.5
    P = np.sign(rng.standard_normal((n, 680)))
    shim = tmp_path / "shim"
    shim.mkdir()
    (shim / "randn.m").write_text("function r = randn(varargin)\nglobal KR_PROBES KR_PROBE_POS\n"
                                  "r = KR_PROBES(:, KR_PROBE_POS + (1:10)); KR_PROBE_POS = KR_PROBE_POS + 10;\nend\n")
    pairs = [(P[:, 20 * k:20 * k + 10], P[:, 20 * k + 10:20 * k + 20]) for k in range(34)]
    maxit = int(rng.choice([30, 60, 90]))
    otr, ores, oit = O.mc_trace(A, n, 1e-3, maxit, 1, 0, probes=pairs)
    I.addpath(str(shim))
    try:
        I.globals["KR_PROBES"], I.globals["KR_PROBE_POS"] = P, np.array([[0.0]])
        tr, res, itr = I.call("mc_trace", sp.csc_matrix(A), n, 1e-3, maxit, 1, 0, nargout=3)
        assert sc(itr) == oit
        close([sc(tr), sc(res)], [otr, ores])
        I.globals["KR_PROBE_POS"] = np.array([[0.0]])
        tre = I.call("trace_exp", sp.csc_matrix(A), nargout=1)[0]
        close(tre, O.trace_exp(A, pairs))
    finally:
        I.rmpath(str(shim))


@pytest.mark.parametrize("seed", range(6))
def test_candidates_and_greedy_random(I, O, seed):
    rng = np.random.default_rng(600 + seed)
    n = int(rng.integers(140, 220))
    A = graph(rng, n, deg=5.0)
    c = rng.uniform(0.1, 1.0, n)
    if seed % 2:
        c = np.round(c, 1)                                   # many TIES in the centrality: the first-match / stable-sort rules decide
    Ac = sp.csc_matrix(A)
    cc = c.reshape(-1, 1)
    num = int(rng.integers(5, 40))
    for order in ("min", "mult"):
        close(I.call("find_top_edges", Ac, cc, num, order, nargout=1)[0], O.find_top_edges(A, c, num, order))
        close(I.call("find_top_missing_edges", Ac, cc, num, order, nargout=1)[0], O.find_top_missing_edges(A, c, num, order))
    miobi = "break" if seed % 2 == 0 else "make"
    rescale = 1.0 if seed % 3 else 2.0
    tol = 1e-7
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        oe, orob, oA = O.greedy_krylov(A, 3, 12, c, "min", tol, 100, np.inf, 0, miobi, rescale)
    e, rob, An = I.call("greedy_krylov", Ac, 3, 12, cc, "min", tol, 100, np.inf, 0, miobi, rescale, nargout=3)
    close(e, oe)
    close(rob, orob)
    assert (sp.csr_matrix(An) != sp.csr_matrix(oA)).nnz == 0
    # krylov_miobi on an explicit list with a self loop and a duplicate row
    E = O.find_top_edges(A, c, 6, "mult").astype(np.float64)
    E[2] = [E[0, 0], E[0, 0]]
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        oe, orob, _ = O.krylov_miobi(A, 2, E.astype(np.int64), tol, 100, np.inf, 0, miobi, rescale)
    e, rob = I.call("krylov_miobi", Ac, 2, E, tol, 100, np.inf, 0, miobi, rescale, nargout=2)
    close(e, oe)
    close(rob, orob)
