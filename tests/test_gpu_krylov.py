"""GPU parity (through the C ABI) of the Krylov evaluators against the oracle on identical inputs.
Tolerance: the north star's 1e-10 relative on fp64 traces / entries / gradients, iteration counts equal."""
import warnings

import numpy as np
import pytest
import scipy.sparse as sp

from conftest import edge_UB

pytestmark = pytest.mark.gpu
RTOL = 1e-10


@pytest.fixture(scope="module")
def kr():
    import krylov_robustness_b200 as kr
    return kr


@pytest.fixture(scope="module")
def O():
    import oracle
    return oracle


def _omega(A, k, seed, min_degree=3):
    L = sp.tril(A, -1).tocoo()
    deg = np.diff(sp.csr_matrix(A).indptr)
    ok = np.where((deg[L.row] >= min_degree) & (deg[L.col] >= min_degree))[0]
    rng = np.random.default_rng(seed)
    sel = ok[rng.choice(ok.size, k, replace=False)]
    return np.stack([L.row[sel] + 1, L.col[sel] + 1], 1), 0.1 * L.data[sel] * rng.random(k)


# ------------------------------------------------------------------ L1
@pytest.mark.parametrize("arnoldi", [False, True])
@pytest.mark.parametrize("bs", [1, 2, 5, 24])
def test_krylov_basis_invariants(kr, O, graphs, arnoldi, bs):
    A = graphs("oregon_A1")
    n = A.shape[0]
    b = np.random.default_rng(bs).standard_normal((n, bs))
    steps = 6
    if arnoldi:
        V, K, H, p, lucky = kr.arnoldi_krylov(A, b)
        oV, oK, oH, op_, _ = O.arnoldi_krylov(A, b)
        for _ in range(steps - 1):
            V, K, H, p, lucky = kr.arnoldi_krylov(V, K, H, p)
            oV, oK, oH, op_, _ = O.arnoldi_krylov(oV, oK, oH, op_)
        assert V.shape == oV.shape and H.shape == oH.shape and np.array_equal(K, oK)
        assert np.linalg.norm(V.T @ V - np.eye(V.shape[1])) < 1e-12
        assert np.linalg.norm(A @ (V @ K) - V @ H) < 1e-10 * np.linalg.norm(H)
    else:
        V, H, p, lucky = kr.lanczos_krylov(A, b)
        oV, oH, op_, _ = O.lanczos_krylov(A, b)
        for _ in range(steps - 1):
            V, H, p, lucky = kr.lanczos_krylov(V, H, p)
            oV, oH, op_, _ = O.lanczos_krylov(oV, oH, op_)
        assert V.shape == (n, 2 * bs) and H.shape == oH.shape
        assert np.linalg.norm(V.T @ V - np.eye(2 * bs)) < 1e-12
        assert np.allclose(p.last, V[:, bs:])
    assert not lucky
    # basis-independent: spectrum of the symmetrised projection (what every caller consumes)
    G = H[:-bs, :]
    oG = oH[:-bs, :]
    ev = np.linalg.eigvalsh((G + G.T) / 2)
    oev = np.linalg.eigvalsh((oG + oG.T) / 2)
    assert np.max(np.abs(ev - oev)) <= RTOL * np.max(np.abs(oev))
    # Householder conventions match LAPACK's, so even the block entries agree up to rounding
    assert np.allclose(np.abs(H), np.abs(oH), rtol=1e-8, atol=1e-10 * np.abs(oH).max())
    # ... SIGNS included: the thin QR is two rounds of Cholesky QR on the tensor cores whose column signs are
    # reconstructed to be those of dgeqr2 / dorg2r (tsdense.cuh::thin_qr), so V and H are the reference's, not just
    # a sign-flipped equivalent
    assert np.allclose(H, oH, rtol=1e-8, atol=1e-10 * np.abs(oH).max())
    assert np.allclose(V, oV, rtol=0, atol=1e-9)


def test_krylov_errors(kr, graphs):
    A = graphs("oregon_A0")
    with pytest.raises(ValueError, match="wrong number of rows"):
        kr.lanczos_krylov(A, np.ones((5, 1)))
    with pytest.raises(ValueError, match="wrong number of arguments"):
        kr.arnoldi_krylov(A)


# ------------------------------------------------------------------ trace_fun_update
@pytest.mark.parametrize("gname,fun,sign", [("oregon_A0", "exp", -1.0), ("oregon_A8", "exp", 1.0),
                                           ("transport_Rome", "sinh", -1.0), ("transport_Barcelona", "cosh", 1.0)])
def test_trace_fun_update_edges_vs_oracle(kr, O, graphs, gname, fun, sign):
    A = graphs(gname)
    n = A.shape[0]
    f = {"exp": np.exp, "sinh": np.sinh, "cosh": np.cosh}[fun]
    nrm, _ = O.normest(A, 1e-2)
    tol = 1e-6 * abs(f(nrm))
    c = O.compute_centrality(A, "eig")
    E = O.find_top_edges(A, c, 24, "min") if sign < 0 else O.find_top_missing_edges(A, c, 24, "min")
    x, it, lucky = kr.trace_fun_update_edges(A, E, sign, tol, 100, fun)
    for h, (i, j) in enumerate(E):
        U, B = edge_UB(n, int(i), int(j), sign)
        ox, oit, olucky = O.trace_fun_update(A, U, B, tol, 100, 0, fun)
        assert it[h] == oit and bool(lucky[h]) == bool(olucky), (h, it[h], oit)
        assert abs(x[h] - ox) <= RTOL * abs(ox), (h, x[h], ox)
    # the single-candidate entry point: U = [e_i e_j], B = [0 b; b 0] is recognised and takes the pair kernels
    U, B = edge_UB(n, int(E[0, 0]), int(E[0, 1]), sign)
    x1, it1, _ = kr.trace_fun_update(A, U, B, tol, 100, 0, fun)
    assert it1 == it[0] and abs(x1 - x[0]) <= RTOL * abs(x[0])
    # the same rank-2 update written with a rotated basis (U Q, Q' B Q) is NOT of that shape and takes the
    # general wide-block path (cuSOLVER QR / eigen-solves): same update matrix, same answer
    th = 0.3
    Q = np.array([[np.cos(th), -np.sin(th)], [np.sin(th), np.cos(th)]])
    Bq = Q.T @ B @ Q
    Bq = 0.5 * (Bq + Bq.T)                       # exactly symmetric (the device path insists on it)
    x2, it2, _ = kr.trace_fun_update(A, np.asarray(U) @ Q, Bq, tol, 100, 0, fun)
    ox2, oit2, _ = O.trace_fun_update(A, np.asarray(U) @ Q, Bq, tol, 100, 0, fun)
    assert it2 == oit2 and abs(x2 - ox2) <= RTOL * abs(ox2)
    assert abs(x2 - x[0]) <= 1e-8 * abs(x[0])


def test_trace_fun_update_edges_slot_reseeding(kr, O, graphs, monkeypatch):
    """The candidate pipeline keeps a fixed number of slots busy and re-seeds a slot as soon as its candidate has
    converged (slots at different step numbers coexist).  With 8 / 24 slots for 96 candidates every slot is
    re-used many times: values, iteration counts and lucky flags must not depend on the slot count, and match
    the oracle."""
    A = graphs("oregon_A8")
    n = A.shape[0]
    nrm, _ = O.normest(A, 1e-2)
    tol = 1e-6 * np.exp(nrm)
    c = O.compute_centrality(A, "eig")
    E = np.concatenate([O.find_top_edges(A, c, 48, "min"), O.find_top_missing_edges(A, c, 48, "min")])
    # default dispatch on this graph (CSR L2-resident): the single-launch path of pairs_small.cuh, one persistent
    # CTA per candidate.  KR_PAIR_SLOTS forces the batched slot pipeline of pairs.cuh.
    small = [kr.trace_fun_update_edges(A, E[:48], -1.0, tol, 100, "exp"),
             kr.trace_fun_update_edges(A, E[48:], 1.0, tol, 100, "exp")]
    ref = None
    for slots in ("8", "24", "4096"):
        monkeypatch.setenv("KR_PAIR_SLOTS", slots)
        res = [kr.trace_fun_update_edges(A, E[:48], -1.0, tol, 100, "exp"),
               kr.trace_fun_update_edges(A, E[48:], 1.0, tol, 100, "exp")]
        if ref is None:
            ref = res
        for (x, it, lk), (x0, it0, lk0) in zip(res, ref):
            assert np.array_equal(it, it0) and np.array_equal(lk, lk0)
            assert np.array_equal(x, x0), np.abs(x - x0).max()      # slot placement does not change the arithmetic
    monkeypatch.delenv("KR_PAIR_SLOTS")
    for (x, it, lk), (x0, it0, lk0) in zip(small, ref):            # same arithmetic, other summation order
        assert np.array_equal(it, it0) and np.array_equal(lk, lk0)
        assert np.all(np.abs(x - x0) <= RTOL * np.abs(x0)), np.abs(x / x0 - 1).max()
    again = kr.trace_fun_update_edges(A, E[:48], -1.0, tol, 100, "exp")
    assert np.array_equal(again[0], small[0][0])                   # bit-reproducible run to run
    for h in range(0, 96, 5):
        sign = -1.0 if h < 48 else 1.0
        U, B = edge_UB(n, int(E[h, 0]), int(E[h, 1]), sign)
        ox, oit, _ = O.trace_fun_update(A, U, B, tol, 100)
        x, it, _ = ref[0 if h < 48 else 1]
        assert it[h % 48] == oit and abs(x[h % 48] - ox) <= RTOL * abs(ox)


def test_trace_fun_update_edges_with_leaf_endpoints(kr, O, graphs):
    """Edges with a degree-1 endpoint: the first Lanczos block of a (leaf, hub) edge has an exactly zero
    column and the reference continues with LAPACK's Householder completion (a coordinate vector,
    see tests/test_oracle_krylov.py::test_lanczos_rank_deficient_block_is_lapack_completion and
    DESIGN.md).  The batched kernels reproduce that convention."""
    A = graphs("oregon_A0")
    n = A.shape[0]
    L = sp.tril(A, -1).tocoo()
    deg = np.diff(A.indptr)
    leafy = np.where((deg[L.row] == 1) | (deg[L.col] == 1))[0]
    other = np.where((deg[L.row] > 1) & (deg[L.col] > 1))[0]
    sel = np.concatenate([leafy[:40], other[:24]])
    assert leafy.size >= 40
    E = np.stack([L.row[sel] + 1, L.col[sel] + 1], 1)
    nrm, _ = O.normest(A, 1e-2)
    tol = 1e-6 * np.exp(nrm)
    x, it, lucky = kr.trace_fun_update_edges(A, E, -1.0, tol, 100, "exp")
    bad = []
    for h, (i, j) in enumerate(E):
        U, B = edge_UB(n, int(i), int(j), -1.0)
        ox, oit, _ = O.trace_fun_update(A, U, B, tol, 100)
        if it[h] != oit or abs(x[h] - ox) > 1e-9 * max(abs(ox), tol):
            bad.append((h, int(i), int(j), x[h], ox, int(it[h]), oit))
    assert not bad, bad[:5]


def test_trace_fun_update_dense_branch_and_self_loop(kr, O, graphs):
    A = graphs("grid_Austria")[:100, :100].tocsr()
    E = np.array([[7, 3], [50, 50], [99, 1]])
    x, it, lucky = kr.trace_fun_update_edges(A, E, 1.0, 1e-12, 100, "exp")
    for h, (i, j) in enumerate(E):
        U, B = edge_UB(100, int(i), int(j), 1.0)
        ox, oit, _ = O.trace_fun_update(A, U, B)
        assert it[h] == 0 == oit
        assert abs(x[h] - ox) <= RTOL * abs(ox) + 1e-13
    # self loop on a graph large enough for the Krylov branch (krylov_miobi.m:88-98)
    A = graphs("oregon_A0")
    x, it, _ = kr.trace_fun_update_edges(A, np.array([[5, 5]]), -1.0, 1e-3, 100, "exp")
    U, B = edge_UB(633, 5, 5, -1.0)
    ox, oit, _ = O.trace_fun_update(A, U, B, 1e-3, 100)
    assert it[0] == oit and abs(x[0] - ox) <= RTOL * abs(ox)


def test_trace_fun_update_edge_set(kr, O, graphs):
    """Tests/test_unweighted_break.m:94-95: edge2low_rank of an edge set, rk up to 20."""
    A = graphs("oregon_A1")
    n = A.shape[0]
    Om, _ = _omega(A, 10, 3)
    U, B = O.edge2low_rank(Om, n)
    nrm, _ = O.normest(A, 1e-2)
    tol = 1e-6 * np.exp(nrm)
    ox, oit, _ = O.trace_fun_update(A, U.toarray(), B, tol)
    x, it, _ = kr.trace_fun_update(A, U.toarray(), B, tol)
    assert it == oit
    # 7e-14 measured (scripts/diag_edge_set_tol.py): with the hand-written wide-block step the device follows the
    # reference's arithmetic closely enough for the contract's 1e-10 here (round 1: 1e-8 with cuBLAS/cuSOLVER orderings).
    # Blocks that turn numerically rank deficient (Oregon A0 with this selection: step 3) are the documented exception -
    # LAPACK normalises rounding noise there and the reference's own value is only defined to ~1e-2
    # (scripts/diag_edge_set_steps.py, DESIGN.md section 2).
    assert abs(x - ox) <= RTOL * abs(ox)


@pytest.mark.parametrize("gname", ["transport_Rome", "oregon_A7", "misc_as_735"])
def test_trace_fun_update_wide_edge_set(kr, O, graphs, gname):
    """Tests/test_unweighted_break_budget.m:89-90,119-120: edge2low_rank of up to 100 edges, i.e. up to 200 selector
    columns in ONE block (here 195 / 162 / 161; round 2 refused blocks beyond 128 columns until the Householder passes
    got a 256-column instantiation).  With blocks this wide the reference orthogonalises against two blocks only and
    its own value is rounding-determined: 0.07 % (Rome) to 14 % (as_735) from the dense truth, and the ORACLE's value on
    as_735 moves by 0.2 % between two hosts (different BLAS threading).  Device and oracle are therefore held to each
    other at 5 % with equal iteration counts (observed 1e-3 .. 1.3e-2); that the call runs at all is the point."""
    import scipy.sparse as sp
    A = graphs(gname)
    n = A.shape[0]
    T = sp.tril(A, -1).tocoo()
    pick = np.sort(np.random.default_rng(5).choice(T.nnz, 100, replace=False))
    E = np.stack([T.row[pick] + 1, T.col[pick] + 1], 1)
    U, B = O.edge2low_rank(E, n)
    assert 128 < U.shape[1] <= 200
    nrm, _ = O.normest(A, 1e-2)
    tol = 1e-6 * np.exp(nrm)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        ox, oit, olk = O.trace_fun_update(A, U.toarray(), B, tol)
        x, it, lk = kr.trace_fun_update(A, U.toarray(), B, tol)
    print(gname, "rk", U.shape[1], "device", x, it, lk, "oracle", ox, oit, olk, "rel", abs(x - ox) / abs(ox))
    assert abs(it - oit) <= 1 and bool(lk) == bool(olk)
    assert abs(x - ox) <= 5e-2 * abs(ox)


# ------------------------------------------------------------------ fun_update / entries / gradients
@pytest.mark.parametrize("fun", ["exp", "cosh"])
def test_fun_update_arnoldi_vs_oracle(kr, O, graphs, fun):
    A = graphs("oregon_A1")
    n = A.shape[0]
    Om, X = _omega(A, 8, 0)
    U, B = O.updates._low_rank_from_omega(X, Om, n)
    nrm, _ = O.normest(A, 1e-2)
    tol = 1e-8 * np.exp(nrm)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        oXm, oit, _, oUm = O.fun_update(A, U, B, fun, tol, 100, 0, want_basis=True)
        Xm, it, lucky, Um = kr.fun_update(A, U, B, fun, tol, 100, 0, nargout=4)
    assert it == oit and Xm.shape == oXm.shape and Um.shape == oUm.shape
    ref = oUm @ oXm @ oUm.T
    got = Um @ Xm @ Um.T
    assert np.linalg.norm(got - ref) <= 1e-9 * np.linalg.norm(ref)
    assert abs(np.trace(Xm) - np.trace(oXm)) <= RTOL * abs(np.trace(oXm))


def test_fun_update_lanczos_and_dense_fallback(kr, O, graphs):
    A = graphs("transport_Rome")
    n = A.shape[0]
    Om, X = _omega(A, 3, 1, min_degree=2)
    U, B = O.updates._low_rank_from_omega(X, Om, n)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        oXm, oit, _, _ = O.fun_update(A, U, B, "exp", 1e-8, 100, 0, want_basis=False)
        Xm, it, _ = kr.fun_update(A, U, B, "exp", 1e-8, 100, 0, nargout=3)
    assert it == oit
    assert np.max(np.abs(np.linalg.eigvalsh((Xm + Xm.T) / 2) - np.linalg.eigvalsh((oXm + oXm.T) / 2))) \
        <= 1e-9 * np.abs(oXm).max()
    # dense fallback once the basis spans half the space (fun_update.m:85-90)
    A = graphs("grid_Austria")
    Om, X = _omega(A, 30, 1, min_degree=1)
    U, B = O.updates._low_rank_from_omega(X, Om, A.shape[0])
    oXm, oit, _, oUm = O.fun_update(A, U, B, "cosh", 1e-10, 100, 0, want_basis=True)
    Xm, it, _, Um = kr.fun_update(A, U, B, "cosh", 1e-10, 100, 0, nargout=4)
    assert it == oit and np.array_equal(Um, np.eye(A.shape[0]))
    assert np.max(np.abs(Xm - oXm)) <= 1e-11 * max(1.0, np.abs(oXm).max())


@pytest.mark.parametrize("gname,fun", [("oregon_A0", "exp"), ("oregon_A0", "cosh"), ("transport_Rome", "sinh")])
def test_function_multiple_entries_vs_oracle(kr, O, graphs, gname, fun):
    A = graphs(gname)
    n = A.shape[0]
    f = {"exp": np.exp, "sinh": np.sinh, "cosh": np.cosh}[fun]
    nrm, _ = O.normest(A, 1e-2)
    rng = np.random.default_rng(5)
    om = np.stack([rng.integers(1, n + 1, 40), rng.integers(1, n + 1, 40)], 1)
    om[5:12, 0] = om[5, 0]                       # several pairs share a row index (:42)
    om[12] = [3, 3]
    tol = 1e-8 * f(nrm)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        oX, oit = O.function_multiple_entries(A, om, fun, tol, 100)
        X, it = kr.function_multiple_entries(A, om, fun, tol, 100)
    assert it == oit
    assert np.max(np.abs(X - oX)) <= RTOL * np.max(np.abs(oX))


@pytest.mark.parametrize("gname,fun,npairs,scale", [
    pytest.param("transport_Vermont", "cosh", 400, 1.0, id="transport_Vermont-cosh-400"),
    pytest.param("transport_Rome", "exp", 120, 1.0, id="transport_Rome-exp-120"),
    pytest.param("grid_England", "sinh", 60, 1.0, id="grid_England-sinh-60"),
    pytest.param("grid_England", "cosh", 60, 20.0, id="grid_England-cosh-60-x20")])
def test_function_multiple_entries_local_vs_dense(kr, O, graphs, monkeypatch, gname, fun, npairs, scale):
    """Spaces whose vectors stay on a small ball around the start node run whole in one CTA (csrc/entries_local.cuh);
    the others (ball or step budget exceeded) take the dense batch.  Both orders of arithmetic follow
    arnoldi_krylov.m:104-106, so the entries agree to rounding, the iteration count exactly, and the oracle to 1e-10.
    On the road network every space is local: no SpMM launch at all.  Scaled by 20, a third of the spaces that finish
    locally end with ||T||_inf > EL_TAYLOR_MAX_S = 48, where the projected solve is the warp QL instead of the Taylor scheme."""
    A = graphs(gname).astype(np.float64)
    A = (A / A.max() * scale).tocsr()
    n = A.shape[0]
    f = {"exp": np.exp, "sinh": np.sinh, "cosh": np.cosh}[fun]
    nrm, _ = O.normest(A, 1e-2)
    tol = 1e-8 * float(f(nrm))
    L = sp.tril(A, -1).tocoo()
    rng = np.random.default_rng(17)
    sel = rng.choice(L.nnz, min(npairs, L.nnz), replace=False)
    om = np.stack([L.row[sel] + 1, L.col[sel] + 1], 1).astype(np.int64)
    om[3] = [om[3, 0], om[3, 0]]                                  # a diagonal entry
    om[4] = [om[0, 0], int(rng.integers(1, n + 1))]               # a far-away second index (zero unless reached)
    ctx = kr.Context.default()
    M = kr.Matrix(A, ctx)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        c0 = ctx.counters()
        X1, it1 = kr.function_multiple_entries(M, om, fun, tol, 100)
        c1 = ctx.counters()
        monkeypatch.setenv("KR_ENTRIES_LOCAL", "0")
        X0, it0 = kr.function_multiple_entries(M, om, fun, tol, 100)
        c2 = ctx.counters()
        monkeypatch.delenv("KR_ENTRIES_LOCAL")
        oX, oit = O.function_multiple_entries(A, om[:10], fun, tol, 100)
    scale = np.max(np.abs(X0))
    assert it1 == it0
    assert np.max(np.abs(X1 - X0)) <= 1e-12 * scale
    assert np.max(np.abs(X1[:10] - oX)) <= RTOL * max(np.max(np.abs(oX)), 1e-300)
    assert c2["spmm_launches"] - c1["spmm_launches"] > 0                                      # the dense batch launches SpMMs
    if gname == "transport_Vermont":
        assert c1["spmm_launches"] - c0["spmm_launches"] == 0                                 # every space was local
    # an iteration cap below the stopping step is final on both paths
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        Xa, ita = kr.function_multiple_entries(M, om[:40], fun, tol, 5)
        monkeypatch.setenv("KR_ENTRIES_LOCAL", "0")
        Xb, itb = kr.function_multiple_entries(M, om[:40], fun, tol, 5)
    assert ita == itb == 5
    assert np.max(np.abs(Xa - Xb)) <= 1e-12 * scale


def test_function_multiple_entries_local_step_limit_goes_dense(kr, O, graphs, monkeypatch):
    """A space that needs more steps than the one-CTA path carries (24) while the caller allows more is handed to the
    dense batch: same entries and the same iteration count (30 here) as the dense batch alone and as the oracle."""
    A = (graphs("transport_Vermont").astype(np.float64) * 6.0).tocsr()
    nrm, _ = O.normest(A, 1e-2)
    tol = 1e-10 * float(np.exp(nrm))
    L = sp.tril(A, -1).tocoo()
    sel = np.random.default_rng(17).choice(L.nnz, 48, replace=False)
    om = np.stack([L.row[sel] + 1, L.col[sel] + 1], 1).astype(np.int64)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        X1, it1 = kr.function_multiple_entries(A, om, "exp", tol, 100)
        monkeypatch.setenv("KR_ENTRIES_LOCAL", "0")
        X0, it0 = kr.function_multiple_entries(A, om, "exp", tol, 100)
        monkeypatch.delenv("KR_ENTRIES_LOCAL")
        X6, it6 = kr.function_multiple_entries(A, om[:6], "exp", tol, 100)
        oX, oit = O.function_multiple_entries(A, om[:6], "exp", tol, 100)
    assert it1 == it0 and it1 > 24
    assert it6 == oit
    assert np.max(np.abs(X1 - X0)) <= 1e-12 * np.max(np.abs(X0))
    assert np.max(np.abs(X6 - oX)) <= RTOL * np.max(np.abs(oX))


def test_function_multiple_entries_local_small_components(kr, O, monkeypatch):
    """Start nodes whose component is exhausted after a few steps (lucky breakdown: the new vector is exactly zero), an
    isolated node, self loops and a pattern-only matrix: the one-CTA path and the dense batch walk through the same
    arithmetic (inverse norm 0 after the breakdown), and both give the oracle's entries."""
    blocks = []
    rng = np.random.default_rng(3)
    for m in (1, 2, 5, 9, 30):                                   # paths of m nodes; the 1-node block is an isolated node
        P = sp.diags([np.ones(m - 1), np.ones(m - 1)], [-1, 1], shape=(m, m)) if m > 1 else sp.csr_matrix((1, 1))
        blocks.append(sp.csr_matrix(P))
    ring = sp.diags([np.ones(39), np.ones(39)], [-1, 1], shape=(40, 40)).tolil()
    ring[0, 39] = ring[39, 0] = 1.0
    ring[7, 7] = 1.0                                             # a self loop
    blocks.append(sp.csr_matrix(ring))
    A = sp.block_diag(blocks).tocsr().astype(np.float64)
    n = A.shape[0]
    om = np.array([[1, 1], [2, 3], [3, 2], [4, 8], [8, 4], [6, 6], [10, 17], [17, 10], [20, 40], [47, 47], [55, 60],
                   [60, 55], [55, 5], [87, 48]], dtype=np.int64)
    assert om.max() <= n
    for W, tag in ((A, "pattern"), (A.multiply(sp.csr_matrix(np.triu(0.5 + rng.random((n, n))) + np.triu(0.5 + rng.random((n, n)), 1).T)).tocsr(), "weighted")):
        W = ((W + W.T) * 0.5).tocsr()
        for fun in ("exp", "cosh"):
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                X1, it1 = kr.function_multiple_entries(W, om, fun, 1e-10, 20)
                monkeypatch.setenv("KR_ENTRIES_LOCAL", "0")
                X0, it0 = kr.function_multiple_entries(W, om, fun, 1e-10, 20)
                monkeypatch.delenv("KR_ENTRIES_LOCAL")
                oX, oit = O.function_multiple_entries(W, om, fun, 1e-10, 20)
            assert np.all(np.isfinite(X1)), (tag, fun)
            assert it1 == it0 == oit, (tag, fun, it1, it0, oit)
            assert np.max(np.abs(X1 - X0)) <= 1e-12 * max(1.0, np.max(np.abs(X0))), (tag, fun)
            assert np.max(np.abs(X1 - oX)) <= RTOL * max(1.0, np.max(np.abs(oX))), (tag, fun)


def test_function_multiple_entries_chunked_rows(kr, O, graphs, monkeypatch):
    """Distinct row indices are processed in chunks on the device; forcing tiny chunks must not change
    a single bit of the entries (every space is independent)."""
    A = graphs("transport_Barcelona")
    n = A.shape[0]
    rng = np.random.default_rng(9)
    om = np.stack([rng.integers(1, n + 1, 70), rng.integers(1, n + 1, 70)], 1)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        X1, it1 = kr.function_multiple_entries(A, om, "exp", 1e-9, 100)
        monkeypatch.setenv("KR_ENTRIES_CHUNK_COLS", "16")
        X2, it2 = kr.function_multiple_entries(A, om, "exp", 1e-9, 100)
        oX, oit = O.function_multiple_entries(A, om, "exp", 1e-9, 100)
    assert it1 == it2 == oit
    assert np.array_equal(X1, X2)
    assert np.max(np.abs(X1 - oX)) <= RTOL * np.max(np.abs(oX))


def test_fun_and_grad_vs_oracle(kr, O, graphs):
    import scipy.linalg as sla
    A = graphs("oregon_A1")
    Ad = A.toarray()
    Om, X = _omega(A, 12, 5)
    eA = sla.expm(Ad)
    eAo = np.array([eA[a - 1, b - 1] for a, b in Om])
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        of, ogr = O.fun_and_grad_krylov_exp(X, A, Om, eAo, 1e-8, 100)
        f, gr = kr.fun_and_grad_krylov_exp(X, A, Om, eAo, 1e-8, 100)
    assert abs(f - of) <= RTOL * abs(of)
    assert np.linalg.norm(gr - ogr) <= RTOL * np.linalg.norm(ogr)
    f0, g0 = kr.fun_and_grad_krylov_exp(np.zeros(12), A, Om, eAo, 1e-8, 100)
    assert f0 == 0 and np.array_equal(g0, -2 * eAo)
    cA = sla.coshm(Ad)
    dfA = np.array([cA[a - 1, b - 1] for a, b in Om])
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        of, ogr = O.fun_and_grad_krylov_fun(X, A, Om, "sinh", "cosh", dfA, 1e-8, 100)
        f, gr = kr.fun_and_grad_krylov_fun(X, A, Om, "sinh", "cosh", dfA, 1e-8, 100)
    # the value goes through the wide-block (rk = 24) Lanczos variant on an UNSCALED graph (||A|| = 28.7, 13 steps):
    # its local-only orthogonalisation (lanczos_krylov.m:88) loses orthogonality and the reference's own value
    # is 3.7x the dense truth here (-8.84e10 against -2.38e10: ghost copies of the top eigenvalues) - a
    # rounding-determined number that no second implementation can reproduce, so only its magnitude is checked.
    # The stable regime the weighted scripts actually run in is test_fun_and_grad_scaled_grid_vs_oracle below.
    assert abs(f - of) <= 0.2 * abs(of)
    assert np.linalg.norm(gr - ogr) <= RTOL * np.linalg.norm(ogr)
    with pytest.raises(ValueError, match="not Hermitian"):
        kr.fun_and_grad_krylov_fun(X, sp.triu(A).tocsr(), Om, "sinh", "cosh", dfA, 1e-8, 100)


@pytest.mark.parametrize("gname,fun,dfun,ftol", [("grid_Mexico", "sinh", "cosh", RTOL), ("grid_England", "cosh", "sinh", 1e-3),
                                                 ("transport_Rome", "sinh", "cosh", 1e-3)])
def test_fun_and_grad_scaled_grid_vs_oracle(kr, O, graphs, gname, fun, dfun, ftol):
    """The call shape of Tests/test_weighted_sinh_lbfgs.m:38-48,207-214: A scaled by A/max(A), 30 modifiable
    edges, tol_param = 1e-6.  The gradient (block Arnoldi, full reorthogonalisation) agrees with the oracle to 1e-10
    on every graph, and so does the objective on the Mexican grid.  On England and Rome the selector blocks are
    massively RANK DEFICIENT (8 of 32 pivots of the first R factor are exactly zero, later ones are 1e-17 noise:
    scripts/diag_wide_R.py): LAPACK's Householder QR then normalises pure rounding noise into a basis vector
    (functions/lanczos_krylov.m:90), the block Lanczos continues with a rounding-determined direction and the
    reference's own objective moves by O(tol) - the per-step values agree to 1e-15 up to the first noise pivot and
    differ by a constant 4.5e-5 / 5e-7 (relative) afterwards (scripts/diag_wide.py).  Same iteration counts."""
    A = graphs(gname)
    A = (A / A.max()).tocsr()
    nrm, _ = O.normest(A, 1e-2)
    c = O.compute_centrality(A, "eig")
    E = O.find_top_edges(A, c, 100, "min")
    f_ = {"sinh": np.sinh, "cosh": np.cosh}
    vals, _ = O.function_multiple_entries(A, E, dfun, 1e-6 * float(f_[dfun](nrm)), 100)
    ind = np.argsort(-vals, kind="stable")[:30]
    Om, dfA = E[ind], vals[ind]
    x = 0.05 * np.ones(30)
    tol = 1e-6 * float(f_[fun](nrm))
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        of, ogr = O.fun_and_grad_krylov_fun(x, A, Om, fun, dfun, dfA, tol, 100)
        f, gr = kr.fun_and_grad_krylov_fun(x, A, Om, fun, dfun, dfA, tol, 100)
    assert np.linalg.norm(gr - ogr) <= (RTOL if ftol == RTOL else 1e-8) * np.linalg.norm(ogr)
    assert abs(f - of) <= ftol * abs(of), (f, of)


def test_normest_vs_oracle(kr, O, graphs):
    for g in ("oregon_A0", "grid_Mexico"):
        A = graphs(g)
        e, c = kr.normest(A, 1e-2)
        oe, oc = O.normest(A, 1e-2)
        assert c == oc and abs(e - oe) <= 1e-12 * oe


# ------------------------------------------------------------------ greedy drivers
@pytest.mark.parametrize("miobi", ["break", "make"])
def test_greedy_krylov_same_edges_as_oracle(kr, O, graphs, miobi):
    A = graphs("transport_Barcelona")
    nrm, _ = O.normest(A, 1e-2)
    c = O.compute_centrality(A, "eig")
    tol = 1e-6 * np.exp(nrm)
    oe, orob, oA = O.greedy_krylov(A, 4, 30, c, "min", tol, 100, np.inf, 0, miobi)
    e, rob, An = kr.greedy_krylov(A, 4, 30, c, "min", tol, 100, np.inf, 0, miobi)
    assert np.array_equal(e, oe)                  # index-identical ranking
    assert abs(rob - orob) <= RTOL * abs(orob)
    assert (An != oA).nnz == 0
    with pytest.raises(ValueError, match="should be symmetric"):
        kr.greedy_krylov(sp.triu(A).tocsr(), 1, 5, c)


def test_krylov_miobi_and_centrality(kr, O, graphs):
    A = graphs("oregon_A0")
    c = kr.compute_centrality(A, "eig")
    oc = O.compute_centrality(A, "eig")
    assert np.max(np.abs(c - oc)) <= 1e-9
    E = O.find_top_edges(A, oc, 12, "mult")
    assert np.array_equal(kr.find_top_edges(A, c, 12, "mult"), E)
    assert np.array_equal(kr.find_top_missing_edges(A, c, 15, "min"), O.find_top_missing_edges(A, oc, 15, "min"))
    nrm, _ = O.normest(A, 1e-2)
    tol = 1e-6 * np.exp(nrm)
    oe, orob, _ = O.krylov_miobi(A, 2, E, tol, 100, np.inf, 0, "break")
    e, rob, _ = kr.krylov_miobi(A, 2, E, tol, 100, np.inf, 0, "break")
    assert np.array_equal(e, oe) and abs(rob - orob) <= RTOL * abs(orob)


def test_gradient_over_all_edges_vs_dense(kr, graphs):
    """Config C2 shape (SURVEY.md N1): weighted road network, gradient of trace(sinh(A + Delta)) w.r.t. EVERY
    edge weight = 2*cosh(A + Delta)_ij, from one Krylov space per distinct row index (chunked on the
    device), against dense ground truth."""
    import scipy.linalg as sla
    A = graphs("transport_Rome")
    n = A.shape[0]
    L = sp.tril(A, -1).tocoo()
    Om = np.stack([L.row + 1, L.col + 1], 1)            # all 4831 edges
    X = 0.1 * L.data * np.random.default_rng(4).random(L.nnz)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        gr = kr.fun_and_grad_all_edges(X, A, Om, "sinh", "cosh", 1e-10, 100)
    D = sp.csr_matrix((X, (Om[:, 0] - 1, Om[:, 1] - 1)), shape=(n, n))
    At = (A + D + D.T).toarray()
    lam, Q = np.linalg.eigh(At)
    C = (Q * np.cosh(lam)) @ Q.T
    true = -2.0 * C[Om[:, 0] - 1, Om[:, 1] - 1]
    assert np.max(np.abs(gr - true)) <= 1e-8 * np.max(np.abs(true))


@pytest.mark.parametrize("gname,fun", [("grid_England", "exp"), ("oregon_A0", "cosh"), ("grid_Mexico", "sinh")])
def test_hessian_callbacks_vs_oracle(kr, O, graphs, gname, fun):
    """Row f3: hessianfcn_exp / hessianfcn_fun over multiple_frechet_eval."""
    A = graphs(gname)
    if gname == "oregon_A0":
        A = (A / 8.0).tocsr()
    Om, X = _omega(A, 9, 2, min_degree=2)
    Om[3] = [Om[0, 0], Om[5, 1]]               # pairs sharing a row space and a column space
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        if fun == "exp":
            oH = O.hessianfcn_exp(X, A, Om, 1e-10, 60)
            H = kr.hessianfcn_exp(X, A, Om, 1e-10, 60)
        else:
            oH = O.hessianfcn_fun(X, A, Om, fun, 1e-10, 60)
            H = kr.hessianfcn_fun(X, A, Om, fun, 1e-10, 60)
    assert H.shape == oH.shape and np.array_equal(H, H.T)
    assert np.max(np.abs(H - oH)) <= RTOL * np.max(np.abs(oH))
