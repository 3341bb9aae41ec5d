"""Edge scores with a value per candidate on the device (kr_trace_fun_update_edges_w, kr_greedy_round_w) against the
oracle (oracle.weighted_edges, itself held to dense truth in tests/test_oracle_edges_w.py): values to 1e-10 relative,
iteration counts and lucky flags equal, on the single-launch path, the batched slot pipeline and the dense branch
(n <= 130).  Uniform values reproduce kr_trace_fun_update_edges_ex bitwise; the weighted greedy driver reproduces the
oracle driver and, on a 0/1 graph, greedy_krylov; pending edits, the screen, replicas, errors, the MEX ops and the
MATLAB wrappers."""
import io
import os
import sys

import numpy as np
import pytest
import scipy.sparse as sp

from conftest import ROOT, load_graph
from test_oracle_edges_w import mixed_candidates

pytestmark = pytest.mark.gpu

F = {"exp": np.exp, "sinh": np.sinh, "cosh": np.cosh}
GRIDS = ["grid_Austria", "grid_England", "grid_Mexico", "grid_Sweden"]


@pytest.fixture(scope="module")
def kr():
    import krylov_robustness_b200 as kr
    return kr


def graph(name):
    return sp.csr_matrix(load_graph(name)).astype(np.float64)


def tol_for(A, fun):
    # 1e-8 f(||A||), as tests/test_gpu_node_removal.py: tighter, the lag-2 test compares differences at rounding level
    import oracle as O
    nrm, _ = O.normest(A, 1e-2)
    return 1e-8 * F[fun](nrm)


def with_zeros(E, d, count=3):
    d = d.copy()
    d[np.flatnonzero(E[:, 0] != E[:, 1])[:count]] = 0.0
    return d


def oracle_scores(A, E, d, tol, it, fun):
    import oracle.weighted_edges as OW
    return OW.trace_fun_update_edges_w(A, E, d, tol, it, fun)


def assert_matches(dev, ref, tol):
    x, it, lk = dev
    xo, ito, lko = ref
    assert np.array_equal(it, ito), (it, ito)
    assert np.array_equal(lk, lko)
    err = np.abs(x - xo)
    # rounding-level scores (a zero value, sinh before the first odd walk) are compared against a floor far below tol
    assert np.all(err <= 1e-10 * np.abs(xo) + 1e-4 * tol), (err / np.maximum(np.abs(xo), 1e-300)).max()


def top_edge_candidates(A, count, seed):
    """The `count` edges of largest centrality product with values of either sign in 0.5 .. 1.5, plus two self loops."""
    import oracle as O
    rng = np.random.default_rng(seed)
    E = O.find_top_edges(A, O.compute_centrality(A, "eig"), count, "mult")
    E = np.vstack([E, [[E[0, 0], E[0, 0]], [E[3, 1], E[3, 1]]]])
    d = rng.choice([-1.0, 1.0], len(E)) * rng.uniform(0.5, 1.5, len(E))
    return E.astype(np.int64), d


@pytest.mark.parametrize("name", GRIDS)
@pytest.mark.parametrize("fun", ["exp", "sinh", "cosh"])
def test_device_matches_oracle_on_power_grids(kr, name, fun):
    A = graph(name)
    E, d = mixed_candidates(A, seed=len(name))
    d = with_zeros(E, d)
    tol = tol_for(A, fun)
    dev = kr.trace_fun_update_edges_w(kr.Matrix(A), E, d, tol, None, fun)
    assert_matches(dev, oracle_scores(A, E, d, tol, None, fun), tol)
    z = d == 0.0
    assert np.all(dev[0][z] == 0.0)


def test_dense_branch_on_a_small_weighted_graph(kr):
    # n <= 130: every candidate takes trace_fun_update_general with its own B (the reference's dense branch, iter 0)
    A = graph("grid_Austria")[:120, :120].tocsr()
    A.eliminate_zeros()
    E, d = mixed_candidates(A, seed=11)
    tol = tol_for(A, "exp")
    dev = kr.trace_fun_update_edges_w(A, E, d, tol, None, "exp")
    assert_matches(dev, oracle_scores(A, E, d, tol, None, "exp"), tol)


@pytest.mark.parametrize("slots", [None, "16"])
def test_oregon_A7_on_both_pipelines(kr, monkeypatch, slots):
    # default: the single-launch path (pairs_small.cuh); KR_PAIR_SLOTS = 16: the batched slot pipeline (pairs.cuh) with
    # 40 candidates re-seeded through 16 slots
    if slots:
        monkeypatch.setenv("KR_PAIR_SLOTS", slots)
    A = graph("oregon_A7")
    E, d = top_edge_candidates(A, 38, seed=2)
    d = with_zeros(E, d, 2)
    tol = tol_for(A, "exp")
    dev = kr.trace_fun_update_edges_w(kr.Matrix(A), E, d, tol, 100, "exp")
    assert_matches(dev, oracle_scores(A, E, d, tol, 100, "exp"), tol)
    again = kr.trace_fun_update_edges_w(kr.Matrix(A), E, d, tol, 100, "exp")
    for u, w in zip(dev, again):
        assert np.array_equal(u, w)


@pytest.mark.parametrize("name,slots", [("oregon_A7", None), ("oregon_A7", "16"), ("grid_Mexico", None),
                                        ("grid_Austria", None)])
@pytest.mark.parametrize("rescale", [1.0, 3.7])
def test_uniform_values_equal_the_scalar_path_bitwise(kr, monkeypatch, name, slots, rescale):
    if slots:
        monkeypatch.setenv("KR_PAIR_SLOTS", slots)
    A = graph(name)
    E, _ = top_edge_candidates(A, 30, seed=4)
    b_off, b_self = -1.0 / rescale, -1.0
    d = np.where(E[:, 0] == E[:, 1], b_self, b_off)
    M = kr.Matrix(A)
    tol = tol_for(A, "cosh")
    ref = kr.trace_fun_update_edges(M, E, b_off, tol, 100, "cosh", b_self=b_self)
    dev = kr.trace_fun_update_edges_w(M, E, d, tol, 100, "cosh")
    for u, w in zip(ref, dev):
        assert np.array_equal(u, w)


def test_pending_edits_score_the_edited_matrix(kr):
    A = graph("grid_England")
    E, d = mixed_candidates(A, seed=9)
    pairs = [(int(i), int(j)) for i, j in E if i != j]
    (a, b), (c, e), (f, g) = pairs[0], pairs[1], pairs[2]
    edits = [(a, b, 0.0),                              # a candidate edge deleted
             (c, e, 0.37),                             # a candidate's weight changed
             (f, int(E[-1, 0]), 0.5),                  # an edge inserted next to a candidate
             (g, g, 0.25)]                             # a diagonal entry
    M = kr.Matrix(A)
    B = A.tolil()
    for i, j, v in edits:
        M.set_edges([i], [j], v)
        B[i - 1, j - 1] = v
        B[j - 1, i - 1] = v
    B = B.tocsr()
    B.eliminate_zeros()
    Bd = B.toarray()
    d = np.array([-Bd[i - 1, j - 1] if (i != j and Bd[i - 1, j - 1] != 0) else dh for (i, j), dh in zip(E, d)])
    tol = tol_for(B, "exp")
    dev = kr.trace_fun_update_edges_w(M, E, d, tol, None, "exp")
    assert_matches(dev, oracle_scores(B, E, d, tol, None, "exp"), tol)


@pytest.mark.parametrize("miobi", ["make", "break"])
def test_screened_weighted_round_selects_the_exact_winner(kr, miobi):
    from krylov_robustness_b200.graphs import power_law_graph, spectral_radius_estimate
    A = power_law_graph(60_000, 1_200_000, 2.2, 7)
    lam = spectral_radius_estimate(A, 30)
    A = (A * (1.0 / lam)).tocsr()
    M = kr.Matrix(A)
    E = kr.find_top_missing_edges(A, kr.compute_centrality(M, "eig"), 3000, "min")
    rng = np.random.default_rng(5)
    d = (1.0 if miobi == "make" else -1.0) * rng.uniform(0.5, 1.5, len(E)) / lam
    tol = 1e-6 * float(np.e)
    x = kr.trace_fun_update_edges_w(M, E, d, tol, 100, "exp")[0]
    b0, v0, s0, m0, i0 = kr.greedy_round_w(M, E, d, tol, 100, "exp", miobi, screen=False)
    assert m0.all() and np.array_equal(s0, x) and i0["screened"] == 0
    assert (b0, v0) == kr.select_candidate(x, miobi)
    b1, v1, s1, m1, i1 = kr.greedy_round_w(M, E, d, tol, 100, "exp", miobi, screen=True)
    assert i1["screened"] > 0.9 * len(E) and i1["exact"] < 0.2 * len(E), i1
    assert (b1, v1) == (b0, v0)
    assert np.array_equal(s1[m1], x[m1])
    assert (np.abs(s1 - x) / np.abs(x)).max() <= 1e-6


@pytest.mark.parametrize("miobi", ["break", "make"])
def test_weighted_greedy_matches_the_oracle_driver(kr, miobi):
    import oracle as O
    import oracle.weighted_edges as OW
    A = graph("grid_England")
    c = O.compute_centrality(A, "eig")
    tol = 1e-8 * np.exp(O.normest(A, 1e-2)[0])
    k, Q = 10, 30
    w = None if miobi == "break" else np.random.default_rng(3).uniform(0.5, 1.5, Q + k)
    order = "mult" if miobi == "break" else "min"
    ed, rd, Ad, ad = kr.greedy_krylov_weighted(A, k, Q, c, order, tol, None, "exp", miobi, w)
    eo, ro, Ao, ao = OW.greedy_krylov_weighted(A, k, Q, c, order, tol, None, "exp", miobi, w)
    assert np.array_equal(ed, eo)
    assert abs(rd - ro) <= 1e-10 * abs(ro)
    assert np.array_equal(ad, ao)
    assert abs(Ad - Ao).max() == 0.0
    if miobi == "break":
        assert np.array_equal(ad, -A.toarray()[ed[:, 0] - 1, ed[:, 1] - 1])    # the grid's own weights were removed
    scr = kr.greedy_krylov_weighted(A, k, Q, c, order, tol, None, "exp", miobi, w, screen=True)
    assert np.array_equal(scr[0], ed) and scr[1] == rd


@pytest.mark.parametrize("miobi,order", [("break", "mult"), ("make", "min")])
def test_weighted_greedy_on_oregon_A0_is_greedy_krylov_bitwise(kr, miobi, order):
    import oracle as O
    A = graph("oregon_A0")
    c = O.compute_centrality(A, "eig")
    tol = 1e-8 * np.exp(O.normest(A, 1e-2)[0])
    e1, r1, A1 = kr.greedy_krylov(A, 5, 40, c, order, tol, None, miobi=miobi)
    e2, r2, A2, applied = kr.greedy_krylov_weighted(A, 5, 40, c, order, tol, None, "exp", miobi)
    assert np.array_equal(e1, e2)
    assert r1 == r2
    assert (A1 != A2).nnz == 0
    assert np.all(applied == (-1.0 if miobi == "break" else 1.0))


def test_replicas_split_the_list_bitwise(kr):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("one GPU")
    A = graph("oregon_A7")
    E, d = top_edge_candidates(A, 62, seed=6)
    tol = tol_for(A, "exp")
    single = kr.trace_fun_update_edges_w(kr.Matrix(A), E, d, tol, 100, "exp")
    multi = kr.Matrix(A)
    assert multi.replicate() >= 2
    shared = kr.trace_fun_update_edges_w(multi, E, d, tol, 100, "exp")
    for u, w in zip(single, shared):
        assert np.array_equal(u, w)


def test_argument_errors(kr):
    import ctypes as C
    A = graph("grid_Sweden")
    n = A.shape[0]
    M = kr.Matrix(A)
    E = np.array([[1, 2], [3, 3]])
    err = kr._lib.KrylovB200Error
    with pytest.raises(err, match="non-finite value d\\(2\\)"):
        kr.trace_fun_update_edges_w(M, E, [1.0, np.nan], 1e-8, 20)
    with pytest.raises(err, match="non-finite value d\\(1\\)"):
        kr.greedy_round_w(M, E, [np.inf, 1.0], 1e-8, 20)
    with pytest.raises(err, match="edge index out of range"):
        kr.trace_fun_update_edges_w(M, [[1, n + 1]], [1.0], 1e-8, 20)
    with pytest.raises(err, match="edge index out of range"):
        kr.greedy_round_w(M, [[0, 2]], [1.0], 1e-8, 20)
    with pytest.raises(err, match="it must be >= 1"):
        kr.trace_fun_update_edges_w(M, E, 1.0, 1e-8, 0)
    with pytest.raises(ValueError, match="unsupported function"):
        kr.trace_fun_update_edges_w(M, E, 1.0, 1e-8, 20, "tanh")
    with pytest.raises(ValueError, match="one value per row of E"):
        kr.trace_fun_update_edges_w(M, E, [1.0, 2.0, 3.0], 1e-8, 20)
    with pytest.raises(ValueError, match="weights must be a scalar or align"):
        kr.greedy_krylov_weighted(A, 2, 10, np.ones(n), "min", 1e-8, 20, "exp", "make", np.ones(3))
    lib = M.ctx.lib
    x = np.zeros(2)
    k = np.zeros(2, dtype=np.int64)
    lk = np.zeros(2, dtype=np.int32)
    Ef = np.asfortranarray(E.astype(np.int64))
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    with pytest.raises(err, match="null argument"):
        kr._lib.check(lib.kr_trace_fun_update_edges_w(M.ctx.h, M.h, 2, p(Ef), None, 1e-8, 20, 0, p(x), p(k), p(lk)))
    x, it, lk = kr.trace_fun_update_edges_w(M, np.zeros((0, 2), dtype=np.int64), np.zeros(0), 1e-8, 20)
    assert x.size == it.size == lk.size == 0


def test_mex_ops_match_the_python_bindings(kr, tmp_path):
    sys.path.insert(0, os.path.join(ROOT, "tests", "mex_stub"))
    import bridge
    H = bridge.MexHost(bridge.build_host(tmp_path))
    A = graph("grid_Mexico")
    E, d = mixed_candidates(A, seed=13)
    tol = tol_for(A, "exp")
    x, it, lk = kr.trace_fun_update_edges_w(A, E, d, tol, 100, "exp")
    out = H.call(["trace_fun_update_edges_w", A, E.astype(float), d[:, None], tol, 100.0, "exp"], 3)
    assert np.array_equal(out[0].ravel(), x)
    assert np.array_equal(out[1].ravel(), it.astype(float))
    assert np.array_equal(out[2].ravel(), lk.astype(float))
    for mode, miobi in ((0, "break"), (1, "make")):
        b, v = kr.greedy_round_w(A, E, d, tol, 100, "exp", miobi, screen=False)[:2]
        out = H.call(["greedy_round_w", A, E.astype(float), d[:, None], tol, 100.0, "exp", float(mode), 0.0], 3)
        assert float(out[0].ravel()[0]) == b + 1 and float(out[1].ravel()[0]) == v and float(out[2].ravel()[0]) == len(E)


def test_matlab_wrappers_through_the_dropin_harness(kr, tmp_path):
    sys.path.insert(0, os.path.join(ROOT, "tests", "mex_stub"))
    import bridge
    from oracle.mlab import Interpreter
    import oracle as O
    H = bridge.MexHost(bridge.build_host(tmp_path))
    I = Interpreter(stdout=io.StringIO())
    H.install(I)
    I.addpath(os.path.join(ROOT, "krylov_robustness_b200", "matlab"))
    A = graph("grid_Sweden")
    Ac = A.tocsc()
    E, d = mixed_candidates(A, seed=17)
    tol = tol_for(A, "cosh")
    x, it, lk = kr.trace_fun_update_edges_w(A, E, d, tol, 100, "cosh")
    got = I.call("trace_fun_update_edges_w", Ac, E.astype(float), d[:, None], tol, 100.0, np.zeros((0, 0)), nargout=3)
    assert H.calls.get("trace_fun_update_edges_w", 0) == 1
    assert got[0].ravel().shape == x.shape
    # fun = [] takes the default @exp in the wrapper: compare with the binding's exp scores
    xe = kr.trace_fun_update_edges_w(A, E, d, tol, 100, "exp")[0]
    assert np.array_equal(got[0].ravel(), xe)
    c = O.compute_centrality(A, "eig")
    k, Q = 4, 20
    for miobi, order, w in (("break", "mult", None), ("make", "min", np.linspace(0.5, 1.5, Q + k))):
        top = (kr.find_top_missing_edges if miobi == "make" else kr.find_top_edges)(A, c, Q + k, order)
        ed, rd, Ad, ad = kr.greedy_krylov_weighted(A, k, Q, c, order, tol, 100, "exp", miobi, w)
        args = [Ac, float(k), float(Q), top.astype(float), tol, 100.0, np.zeros((0, 0)), miobi]
        if w is not None:
            args.append(w[:, None])
        em, rm, Am, am = I.call("greedy_krylov_weighted", *args, nargout=4)
        assert np.array_equal(np.asarray(em, dtype=np.int64), ed)
        assert float(np.asarray(rm).ravel()[0]) == rd
        assert np.array_equal(np.asarray(am).ravel(), ad)
        assert abs(sp.csr_matrix(Am) - Ad).max() == 0.0
