"""The SLQ pass returns the same bits whichever way its probes arrive.

The same Rademacher values go in four ways: a device block filled by kr_dense_fill_rademacher (it carries an int8 sign
panel, so step 0 gathers signs and steps 0 and 1 read them), the same values uploaded as fp64 (kr_dense_upload: no
sign panel, the fp64 path), int8 host probes (kr_slq_trace_sign, laid out as a sign panel) and fp64 host probes
(kr_slq_trace).  vals, alpha and beta must agree to the bit, with and without alpha / beta asked for (the last step
then skips its update), for m = 1 (step 0 is also the last step), 2, 3 and 30, k not a multiple of the 16-column
panel, pattern-only and valued A, pending edge edits, and a graph on which every probe breaks down.  The pass
only reads its probe block, and a write into a block drops its sign panel."""
import ctypes as C

import numpy as np
import pytest
import scipy.sparse as sp

pytestmark = pytest.mark.gpu

N = 6_000
K = 37                       # two whole panels and a partial one
SEED = 11


@pytest.fixture(scope="module")
def kr():
    import krylov_robustness_b200 as kr
    return kr


@pytest.fixture(scope="module")
def ctx(kr):
    return kr.Context.default(0)


def _power_law(n, seed, valued):
    """Symmetric graph with rows of every SpMM lane class, two hubs of >= 1024 nonzeros (whole-CTA rows) and
    isolated nodes; scaled so that ||A|| is O(1)."""
    rng = np.random.default_rng(seed)
    deg = np.minimum((rng.pareto(1.6, n) + 1) * 2, 400).astype(int)
    deg[:2] = 1500
    deg[-50:] = 0
    rows = np.repeat(np.arange(n), deg)
    cols = rng.integers(0, n - 50, rows.size)
    keep = rows != cols
    A = sp.coo_matrix((np.ones(keep.sum()), (rows[keep], cols[keep])), shape=(n, n)).tocsr()
    A.data[:] = 1.0
    A = ((A + A.T) > 0).astype(np.float64).tocsr()
    if valued:
        A = sp.triu(A, 1).tocsr()
        A.data = rng.uniform(0.5, 1.5, A.nnz)
        A = (A + A.T).tocsr()
    return A * (1.0 / 60.0)


def _breakdown_graph(n):
    """Disjoint edges and triangles plus isolated nodes: A has four distinct eigenvalues, so every Lanczos run
    breaks down (beta = 0 up to rounding) within four steps."""
    blocks, i = [], 0
    while i + 3 <= n - 100:
        size = 2 if (i // 5) % 2 else 3
        blocks.append(np.ones((size, size)) - np.eye(size))
        i += size
    blocks.append(sp.csr_matrix((n - i, n - i)))
    return sp.block_diag(blocks, format="csr") * 0.5


def _slq(kr, M, Z, m, want_ab, k):
    """One call of the entry point that matches Z; returns (tr, vals, alpha, beta) with alpha / beta None unless
    asked for."""
    lib, ctx = M.ctx.lib, M.ctx
    tr = C.c_double()
    vals = np.full(k, np.nan)
    al = np.full((m, k), np.nan, order="F") if want_ab else None
    be = np.full((m, k), np.nan, order="F") if want_ab else None
    p = lambda a: None if a is None else C.c_void_p(a.ctypes.data)
    if isinstance(Z, kr.Dense):
        rc = lib.kr_slq_trace_dev(ctx.h, M.h, Z.h, m, 0, C.byref(tr), p(vals), p(al), p(be))
    else:
        Zc = np.asfortranarray(Z)
        entry = lib.kr_slq_trace_sign if Zc.dtype == np.int8 else lib.kr_slq_trace
        rc = entry(ctx.h, M.h, k, p(Zc), Zc.shape[0], m, 0, C.byref(tr), p(vals), p(al), p(be))
    assert rc == 0, lib.kr_last_error()
    return tr.value, vals, al, be


def _bits(a):
    return np.ascontiguousarray(a).view(np.int64)


def _same(a, b):
    return a.shape == b.shape and np.array_equal(_bits(a), _bits(b))


def _four_ways(kr, ctx, M, n, k, m, seed=SEED):
    Zh = kr.rademacher_host(n, k, seed)
    Zs = kr.Dense(n, k, ctx).fill_rademacher(seed)
    Zf = kr.Dense(n, k, ctx).upload(Zh)
    inputs = {"sign panel": Zs, "fp64 block": Zf, "int8 host": Zh.astype(np.int8), "fp64 host": Zh}
    out = {}
    for ab in (True, False):
        for name, Z in inputs.items():
            out[name, ab] = _slq(kr, M, Z, m, ab, k)
    return Zh, Zs, Zf, out


def _check_identical(out, m, finite=True):
    ref = out["fp64 host", True]
    for (name, ab), (tr, vals, al, be) in out.items():
        assert _same(vals, ref[1]), (name, ab)
        assert np.float64(tr).view(np.int64) == np.float64(ref[0]).view(np.int64), (name, ab)
        if ab:
            assert _same(al, ref[2]), (name, "alpha")
            assert _same(be, ref[3]), (name, "beta")       # beta_{m-1} included: the norm-only last update
    if finite:
        assert np.all(np.isfinite(ref[1])) and np.all(np.isfinite(ref[3][m - 1]))


@pytest.mark.parametrize("valued", [False, True], ids=["pattern", "valued"])
@pytest.mark.parametrize("m", [1, 2, 3, 30])
def test_sign_and_fp64_probes_agree_bitwise(kr, ctx, valued, m):
    import oracle
    A = _power_law(N, 3, valued)
    M = kr.Matrix(A, ctx)
    assert M.info()["pattern_only"] == (not valued)
    Zh, Zs, Zf, out = _four_ways(kr, ctx, M, N, K, m)
    _check_identical(out, m)
    tr, vals, al, be = oracle.slq_trace(A, Zh, m, "exp")
    got = out["fp64 host", True]
    assert np.allclose(got[1], vals, rtol=1e-9, atol=0)
    assert np.allclose(got[2][:3], al[:3], rtol=1e-9, atol=1e-12)


def test_pending_edits(kr, ctx):
    import oracle
    A = _power_law(N, 5, True)
    M = kr.Matrix(A, ctx)
    rng = np.random.default_rng(7)
    i = rng.integers(0, N, 60)
    j = rng.integers(0, N, 60)
    j[:5] = 0                                          # edits in a hub row (whole-CTA tile)
    v = rng.uniform(0.0, 0.05, 60)
    v[:10] = 0.0                                       # removals
    M.set_edges(i + 1, j + 1, v)                      # symmetric A, few edits: kept pending (the SpMM's DELTA flavour)
    B = A.tolil()
    for a, b, x in zip(i, j, v):
        B[a, b] = x
        B[b, a] = x
    B = B.tocsr()
    B.eliminate_zeros()
    Zh, _, _, out = _four_ways(kr, ctx, M, N, K, 30)
    _check_identical(out, 30)
    assert np.allclose(out["fp64 host", True][1], oracle.slq_trace(B, Zh, 30, "exp")[1], rtol=1e-9, atol=0)


@pytest.mark.parametrize("m", [5, 30])
def test_breakdown(kr, ctx, m):
    A = _breakdown_graph(N)
    M = kr.Matrix(A, ctx)
    _, _, _, out = _four_ways(kr, ctx, M, N, K, m)
    _check_identical(out, m, finite=False)
    assert np.all(np.abs(out["fp64 host", True][3][3]) < 1e-10)


def test_probe_block_is_read_only(kr, ctx):
    A = _power_law(N, 3, False)
    M = kr.Matrix(A, ctx)
    Zh = kr.rademacher_host(N, K, SEED)
    Zs = kr.Dense(N, K, ctx).fill_rademacher(SEED)
    Zf = kr.Dense(N, K, ctx).upload(Zh)
    first = [_slq(kr, M, Z, 30, False, K) for Z in (Zs, Zf)]
    assert _same(Zs.download(), Zh) and _same(Zf.download(), Zh)
    again = [_slq(kr, M, Z, 30, False, K) for Z in (Zs, Zf)]
    for a, b in zip(first, again):
        assert _same(a[1], b[1])


def test_writes_drop_the_sign_panel(kr, ctx):
    A = _power_law(N, 3, False)
    M = kr.Matrix(A, ctx)
    X = np.random.default_rng(2).standard_normal((N, K))
    # upload into a filled block: the pass must see the uploaded values, not the old signs
    Z = kr.Dense(N, K, ctx).fill_rademacher(SEED)
    Z.upload(X)
    fresh = kr.Dense(N, K, ctx).upload(X)
    assert _same(_slq(kr, M, Z, 30, True, K)[1], _slq(kr, M, fresh, 30, True, K)[1])
    # kr_spmm_dev into a filled block
    Y = kr.Dense(N, K, ctx).fill_rademacher(SEED)
    Xd = kr.Dense(N, K, ctx).upload(X)
    assert ctx.lib.kr_spmm_dev(ctx.h, M.h, Xd.h, Y.h) == 0, ctx.lib.kr_last_error()
    Yh = Y.download()
    assert np.allclose(Yh, A @ X, rtol=1e-12, atol=1e-12)
    fresh = kr.Dense(N, K, ctx).upload(Yh)
    assert _same(_slq(kr, M, Y, 30, True, K)[1], _slq(kr, M, fresh, 30, True, K)[1])
    # and a refill brings the sign path back with the new values
    Y.fill_rademacher(SEED + 1)
    ref = kr.Dense(N, K, ctx).upload(kr.rademacher_host(N, K, SEED + 1))
    assert _same(_slq(kr, M, Y, 30, True, K)[1], _slq(kr, M, ref, 30, True, K)[1])
