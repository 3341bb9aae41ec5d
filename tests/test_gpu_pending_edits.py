"""Pending edge edits (kr_matrix_set_edges) against a plain SciPy restatement of the edited matrix.

An edit A(i,j) = A(j,i) = v does not rebuild the device CSR: the host keeps (new value - stored value) per entry and
the SpMM (its DELTA flavour), the candidate seeds of pairs.cuh / pairs_small.cuh and the node screen add those entries
on the fly.  Every other entry point folds them in first, and an unsymmetric matrix or more than 8192 pending entries
take the rebuild at once.  Each test here applies the same edits, in order, to a SciPy copy (MATLAB semantics: the
later edit of a pair wins, 0 removes the entry) and compares the device with that copy or with the oracle run on it.

Values are dyadic and the SpMM inputs small integers, so every product and partial sum is exact in fp64 and the SpMM
must agree bitwise, whatever its summation order."""
import warnings

import numpy as np
import pytest
import scipy.sparse as sp

from conftest import edge_UB, load_graph

pytestmark = pytest.mark.gpu

N = 12_000
KS = (1, 5, 16, 17, 40)                     # the SpMM panel is 16 columns wide: partial, whole and split panels
DELTA_BYTES_PER_ENTRY = 20                  # stored position, row in tile, column (int32 each) and the fp64 delta


@pytest.fixture(scope="module")
def kr():
    import krylov_robustness_b200 as kr
    return kr


@pytest.fixture(scope="module")
def O():
    import oracle
    return oracle


# ------------------------------------------------------------------ the graphs
def _synthetic_pattern():
    """Symmetric graph, n = 12 000: isolated nodes, rows of every SpMM lane class (1-15, 16-63, 64-255, 256-1023),
    two hubs of degree 1024-4096 (one CTA per row) and one above 4096 (staged in chunks of SPMM_CAP)."""
    rng = np.random.default_rng(20261021)
    n = N
    perm = rng.permutation(n)
    isolated = np.sort(perm[:40])
    hubs = [int(perm[40]), int(perm[41]), int(perm[42])]
    targets = [(h, d) for h, d in zip(hubs, (5200, 1500, 3000))]
    targets += [(int(v), int(rng.integers(300, 900))) for v in perm[43:51]]
    targets += [(int(v), int(rng.integers(80, 240))) for v in perm[51:71]]
    targets += [(int(v), int(rng.integers(20, 60))) for v in perm[71:131]]
    pool = perm[131:]
    # Chung-Lu base among the pool: degrees from a handful to a few dozen, some leaves and some isolated by chance
    w = np.exp(rng.normal(0.0, 0.9, pool.size))
    p = w / w.sum()
    m = 7 * pool.size
    u = pool[rng.choice(pool.size, m, p=p)]
    v = pool[rng.choice(pool.size, m, p=p)]
    rows, cols = [u], [v]
    for node, d in targets:
        nb = pool[rng.choice(pool.size, d, replace=False)]
        rows.append(np.full(d, node))
        cols.append(nb)
    r = np.concatenate(rows)
    c = np.concatenate(cols)
    keep = r != c
    r, c = r[keep], c[keep]
    A = sp.csr_matrix((np.ones(2 * r.size), (np.concatenate([r, c]), np.concatenate([c, r]))), shape=(n, n))
    A.sum_duplicates()
    A.data[:] = 0.25                        # pattern-only storage with uval != 1
    return A, isolated, hubs


def _valued_from(A, seed):
    """Same pattern, dyadic weights k/8 (k = +-1..+-16, symmetric) and a few diagonal entries."""
    rng = np.random.default_rng(seed)
    U = sp.triu(A, 1).tocoo()
    k = rng.integers(1, 17, U.nnz) * rng.choice([-1, 1], U.nnz)
    W = sp.csr_matrix((k / 8.0, (U.row, U.col)), shape=A.shape)
    deg = np.diff(A.indptr)
    diag_nodes = rng.choice(np.where(deg > 0)[0], 30, replace=False)
    D = sp.csr_matrix((rng.integers(1, 17, 30) * rng.choice([-1, 1], 30) / 8.0, (diag_nodes, diag_nodes)), shape=A.shape)
    V = (W + W.T + D).tocsr()
    V.sort_indices()
    return V


def _lane_class(length):
    return np.select([length == 0, length < 16, length < 64, length < 256, length < 1024, length <= 4096],
                     [0, 1, 2, 3, 4, 5], 6)


@pytest.fixture(scope="module")
def synth():
    A, isolated, hubs = _synthetic_pattern()
    V = _valued_from(A, 5)
    for M in (A, V):
        cls = _lane_class(np.diff(M.indptr))
        counts = np.bincount(cls, minlength=7)
        assert counts[0] >= 40 and np.all(counts[1:5] > 0), counts      # isolated rows and every lane class
        assert counts[5] == 2 and counts[6] == 1, counts                  # two CTA-per-row hubs, one above SPMM_CAP
        assert M.nnz <= 400_000                                           # pair_small_kernel stays eligible
        assert abs(M - M.T).nnz == 0
    assert A.nnz >= 200_000
    assert V.diagonal().nonzero()[0].size == 30
    return dict(pattern=A, valued=V, isolated=isolated, hubs=hubs)


# ------------------------------------------------------------------ edits
def apply_edits(A, calls):
    """The SciPy restatement: A(i,j) = A(j,i) = v for every edit, in order; 0 removes the entry."""
    L = A.tolil(copy=True)
    for call in calls:
        for i, j, v in call:
            L[i, j] = v
            L[j, i] = v
    B = L.tocsr()
    B.eliminate_zeros()
    B.sort_indices()
    return B


def set_edges(M, call):
    """Runs one set_edges call (0-based edits); returns the bytes it shipped to the device."""
    e = np.asarray(call, dtype=np.float64).reshape(-1, 3)
    h0 = M.ctx.counters()["h2d_bytes"]
    M.set_edges(e[:, 0].astype(np.int64) + 1, e[:, 1].astype(np.int64) + 1, e[:, 2])
    return M.ctx.counters()["h2d_bytes"] - h0


def delta_bytes_bound(n_entries, n):
    """What the delta path ships at most: DELTA_BYTES_PER_ENTRY per pending entry plus one int per tile (<= n + 1)."""
    return DELTA_BYTES_PER_ENTRY * n_entries + 4 * (n + 2)


def _stored_neighbour(A, r, rng, exclude=()):
    nb = [int(c) for c in A.indices[A.indptr[r]:A.indptr[r + 1]] if c != r and c not in exclude]
    return nb[int(rng.integers(len(nb)))]


def _missing_partner(A, r, rng, candidates):
    row = set(A.indices[A.indptr[r]:A.indptr[r + 1]].tolist())
    for c in rng.permutation(candidates):
        if int(c) != r and int(c) not in row:
            return int(c)
    raise AssertionError("no missing partner")


def edit_script(A, isolated, hubs, seed, unit):
    """Two set_edges calls that reach every case of the delta bookkeeping; values are multiples of `unit`/4 (dyadic).
    Returns (calls, tags): tags name the pairs the candidate tests score."""
    rng = np.random.default_rng(seed)
    n = A.shape[0]
    deg = np.diff(A.indptr)
    cls = _lane_class(deg)
    offd = lambda r: int(np.count_nonzero(A.indices[A.indptr[r]:A.indptr[r + 1]] != r))
    val = lambda i, j: float(A[i, j])
    c1, c2 = [], []
    tags = dict(deleted=[], inserted=[], changed=[])
    used = set(hubs) | set(isolated.tolist())
    # deletions of stored entries: one row of every lane class and every hub row
    rows = [int(rng.choice([r for r in np.where(cls == c)[0] if offd(r) >= 3 and r not in used])) for c in (1, 2, 3, 4)]
    rows += hubs
    for r in rows:
        s = _stored_neighbour(A, r, rng, used)
        c1.append((r, s, 0.0))
        tags["deleted"].append((r, s))
        used |= {r, s}
    # insertions: hub <-> isolated, isolated <-> isolated, and missing pairs on every lane class / hub row
    iso = [int(x) for x in isolated[:6]]
    c1 += [(hubs[0], iso[0], 0.75 * unit), (hubs[1], iso[1], unit), (iso[2], iso[3], -0.5 * unit)]
    tags["inserted"] += [(hubs[0], iso[0]), (hubs[1], iso[1])]
    for r in rows:
        s = _missing_partner(A, r, rng, np.where(deg >= 2)[0])
        c1.append((r, s, unit if len(c1) % 2 else 1.25 * unit))
        tags["inserted"].append((r, s))
    # value changes of stored entries (one to a negative value)
    for r in rows[:4]:
        s = _stored_neighbour(A, r, rng, used)
        c1.append((r, s, -0.75 * unit if r == rows[0] else val(r, s) + 0.5 * unit))
        tags["changed"].append((r, s))
        used.add(s)
    # a self loop and, if there is one, the deletion of a stored diagonal entry
    loop = int(rng.choice([r for r in np.where(cls == 2)[0] if A[r, r] == 0 and r not in used]))
    c1.append((loop, loop, 1.5 * unit))
    diag = np.where(A.diagonal() != 0)[0]
    if diag.size:
        c1.append((int(diag[0]), int(diag[0]), 0.0))
    # two end points with an edit to the same third node: the cross term of the seed's Gram (candidate (a, b))
    t = int(rng.choice([r for r in np.where(cls == 1)[0] if r not in used]))
    a, b = [int(x) for x in rng.choice([r for r in np.where((cls == 1) | (cls == 2))[0] if r not in used and r != t
                                        and A[r, t] == 0], 2, replace=False)]
    c1 += [(a, t, 0.5 * unit), (b, t, 0.75 * unit)]
    tags["third"] = (a, b, t)
    # the same pair twice in one call, and again in the next one
    twice = (rows[1], _missing_partner(A, rows[1], rng, np.where(deg >= 2)[0]))
    c1 += [(twice[0], twice[1], 0.25 * unit), (twice[0], twice[1], 1.75 * unit)]
    # a stored pair changed in the first call and set back to its stored value in the second (cancels its entries)
    back = (rows[2], _stored_neighbour(A, rows[2], rng, used))
    c1.append((back[0], back[1], val(*back) + unit))
    c2 += [(twice[1], twice[0], 0.5 * unit), (back[1], back[0], val(*back))]
    tags["back"] = back
    # second call: more edits on the hub rows (both orientations) and an isolated pair
    for h in hubs:
        s = _stored_neighbour(A, h, rng, used)
        c2.append((s, h, 0.0) if s < h else (h, s, 0.0))
        tags["deleted"].append((h, s))
    c2.append((iso[4], iso[5], 0.5 * unit))
    if unit == A.data[0] and np.all(A.data == A.data[0]):
        # pattern-only storage: an insertion at exactly the stored value and one elsewhere
        r = rows[0]
        c2 += [(r, _missing_partner(A, r, rng, np.arange(n)), unit), (r, _missing_partner(A, r, rng, np.arange(n)), 3 * unit)]
    return [c1, c2], tags


def int_block(n, k, seed):
    return np.random.default_rng(seed).integers(-3, 4, (n, k)).astype(np.float64)


def assert_spmm_exact(kr, M, A, seed, ks=KS):
    """M @ X and kr_spmm_dev agree bitwise with SciPy for small-integer X."""
    n = A.shape[0]
    for k in ks:
        X = int_block(n, k, seed + k)
        ref = A @ X
        Y = M @ X
        assert np.array_equal(Y, ref), (k, np.abs(Y - ref).max())
    X = int_block(n, 17, seed)
    D, Dy = kr.Dense(n, 17, M.ctx).upload(X), kr.Dense(n, 17, M.ctx)
    kr._lib.check(M.ctx.lib.kr_spmm_dev(M.ctx.h, M.h, D.h, Dy.h))
    assert np.array_equal(Dy.download(), A @ X)


def _info_matches(M, A):
    info = M.info()
    assert info["nnz"] == A.nnz, (info["nnz"], A.nnz)
    assert info["nonnegative"] == bool(np.all(A.data >= 0))
    assert info["symmetric"] == (abs(A - A.T).nnz == 0)
    return info


# ------------------------------------------------------------------ 1. SpMM
@pytest.mark.parametrize("variant", ["pattern", "valued"])
def test_spmm_exact_after_edits(kr, synth, variant):
    A0 = synth[variant]
    n = A0.shape[0]
    unit = 0.25 if variant == "pattern" else 0.125
    calls, _ = edit_script(A0, synth["isolated"], synth["hubs"], 1, unit)
    M = kr.Matrix(A0)
    assert M.info()["pattern_only"] == (variant == "pattern")
    edits = 0
    for step, call in enumerate(calls):
        shipped = set_edges(M, call)
        edits += len(call)
        assert shipped <= delta_bytes_bound(2 * edits, n), shipped       # the delta path, not a rebuild ...
        assert shipped < 4 * A0.nnz                                     # ... which ships the whole CSR
        A = apply_edits(A0, calls[:step + 1])
        assert_spmm_exact(kr, M, A, 10 * step)
    X = np.random.default_rng(3).standard_normal((n, 21))
    Y = M @ X
    assert np.abs(Y - A @ X).max() <= 1e-14 * (abs(A) @ np.abs(X)).max()
    assert M.info()["pattern_only"] == (variant == "pattern")           # a property of the storage


def test_edits_that_cancel(kr, synth):
    A0 = synth["valued"]
    calls, _ = edit_script(A0, synth["isolated"], synth["hubs"], 2, 0.125)
    M = kr.Matrix(A0)
    set_edges(M, calls[0])
    A1 = apply_edits(A0, calls[:1])
    assert_spmm_exact(kr, M, A1, 0, ks=(5,))
    undo = [(i, j, float(A0[i, j])) for i, j, _ in calls[0]]            # every touched pair back to its stored value
    shipped = set_edges(M, undo)
    assert shipped <= delta_bytes_bound(0, A0.shape[0])                 # nothing is pending any more
    assert_spmm_exact(kr, M, A0, 1)
    _info_matches(M, A0)


# ------------------------------------------------------------------ 2. the 8192-entry switch
def _new_pairs(A, count, seed):
    rng = np.random.default_rng(seed)
    n = A.shape[0]
    have = set()
    out = []
    while len(out) < count:
        i, j = (int(x) for x in rng.integers(0, n, 2))
        if i == j or (min(i, j), max(i, j)) in have or A[i, j] != 0:
            continue
        have.add((min(i, j), max(i, j)))
        out.append((i, j, 0.25 * float(rng.integers(1, 8))))
    return out


@pytest.mark.parametrize("variant", ["pattern", "valued"])
def test_pending_limit_switches_to_rebuild(kr, synth, variant):
    A0 = synth[variant]
    n = A0.shape[0]
    assert A0.nnz >= 200_000
    pairs = _new_pairs(A0, 4097, 7)
    # 4096 off-diagonal pairs = 8192 pending entries: still the delta path
    M = kr.Matrix(A0)
    shipped = set_edges(M, pairs[:4096])
    assert shipped <= delta_bytes_bound(8192, n) < 4 * A0.nnz, shipped
    assert_spmm_exact(kr, M, apply_edits(A0, [pairs[:4096]]), 20, ks=(5, 17))
    # 4097 pairs = 8194 entries: the host folds them into a new CSR and uploads all of it
    M = kr.Matrix(A0)
    shipped = set_edges(M, pairs)
    A1 = apply_edits(A0, [pairs])
    assert shipped >= 4 * A1.nnz, shipped
    assert_spmm_exact(kr, M, A1, 30, ks=(5, 17))
    _info_matches(M, A1)
    # later edits are relative to the rebuilt matrix: delete some of the new pairs, change others, and set the last
    # one to the value it now has (nothing pending)
    more = [(i, j, 0.0) for i, j, _ in pairs[:5]] + [(i, j, -0.5) for i, j, _ in pairs[5:9]] + pairs[-1:]
    shipped = set_edges(M, more)
    assert shipped <= delta_bytes_bound(2 * len(more), n)
    A2 = apply_edits(A1, [more])
    assert_spmm_exact(kr, M, A2, 40, ks=(1, 17))
    _info_matches(M, A2)


# ------------------------------------------------------------------ 3. folding interleaved with pending edits
def _pow2_scale(O, A):
    """A power of two that brings the spectral radius near 1 and keeps every value dyadic."""
    nrm, _ = O.normest(A, 1e-2)
    return 2.0 ** -np.round(np.log2(nrm))


def test_interleaved_folding(kr, O, synth):
    """Pending edits, a fold (normest), more pending edits on top of the folded matrix, then an entry point that folds
    again (function_multiple_entries): the SpMM is exact at every stage and the entries match the oracle."""
    A0 = synth["valued"]
    s = _pow2_scale(O, A0)
    As = (A0 * s).tocsr()
    calls, tags = edit_script(A0, synth["isolated"], synth["hubs"], 3, 0.125)
    calls = [[(i, j, v * s) for i, j, v in c] for c in calls]
    M = kr.Matrix(As)
    set_edges(M, calls[0])
    A1 = apply_edits(As, calls[:1])
    assert_spmm_exact(kr, M, A1, 0, ks=(5, 17))
    e, c = kr.normest(M, 1e-2)                                          # folds the edits in
    oe, oc = O.normest(A1, 1e-2)
    assert c == oc and abs(e - oe) <= 1e-12 * oe
    assert_spmm_exact(kr, M, A1, 1, ks=(5, 17))
    set_edges(M, calls[1])                                              # relative to the folded matrix
    A2 = apply_edits(As, calls)
    assert_spmm_exact(kr, M, A2, 2, ks=(5, 17))
    _info_matches(M, A2)
    rng = np.random.default_rng(4)
    tri = sp.triu(A2, 0).tocoo()
    pick = rng.choice(tri.nnz, 10, replace=False)
    om = np.stack([tri.row[pick] + 1, tri.col[pick] + 1], 1).astype(np.int64)
    a, b, t = tags["third"]
    h = synth["hubs"][0]
    om = np.concatenate([om, [[a + 1, b + 1], [t + 1, t + 1], [h + 1, h + 1], [h + 1, tags["inserted"][0][1] + 1]]])
    nrm, _ = O.normest(A2, 1e-2)
    tol = 1e-8 * np.exp(nrm)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        oX, oit = O.function_multiple_entries(A2, om, "exp", tol, 100)
        X, it = kr.function_multiple_entries(M, om, "exp", tol, 100)
    assert it == oit
    assert np.max(np.abs(X - oX)) <= 1e-10 * np.max(np.abs(oX))


# ------------------------------------------------------------------ 4. SLQ
def test_slq_after_edits(kr, O, synth):
    A0 = synth["valued"]
    s = _pow2_scale(O, A0)
    As = (A0 * s).tocsr()
    calls, _ = edit_script(A0, synth["isolated"], synth["hubs"], 5, 0.125)
    calls = [[(i, j, v * s) for i, j, v in c] for c in calls]
    M = kr.Matrix(As)
    for c in calls:
        set_edges(M, c)
    A = apply_edits(As, calls)
    n = A.shape[0]
    Z = kr.rademacher_host(n, 24, 9)
    otr, ovals, oal, obe = O.slq_trace(A, Z, 20, "exp")
    Zs = np.asfortranarray(Z.astype(np.int8))
    for probes in (Z, Zs):                                  # kr_slq_trace (fp64 probes), kr_slq_trace_sign (int8)
        tr, vals, al, be = kr.slq_trace(M, probes, 20, "exp", return_details=True)
        assert abs(tr - otr) <= 1e-10 * abs(otr)
        assert np.max(np.abs(vals - ovals)) <= 1e-10 * np.max(np.abs(ovals))
        assert np.max(np.abs(al - oal)) <= 1e-9 * np.max(np.abs(oal))
        assert np.max(np.abs(be - obe)) <= 1e-9 * np.max(np.abs(obe))
    assert_spmm_exact(kr, M, A, 50, ks=(5,))                # the edits are still pending (nothing folded them)


# ------------------------------------------------------------------ 5. candidate scores
def _special(A, E):
    """Rank-deficient first blocks (a leaf end point; adjacent twins): the documented LAPACK-completion cases."""
    deg = np.diff(A.indptr)
    nbr = lambda v: set(A.indices[A.indptr[v]:A.indptr[v + 1]].tolist()) | {v}
    return np.array([deg[i - 1] <= 1 or deg[j - 1] <= 1 or (i != j and nbr(i - 1) == nbr(j - 1)) for i, j in E])


def _candidate_lists(A, tags, hubs, rng):
    """1-based candidates on the EDITED matrix A: (existing edges to break, missing edges to make).  They are the
    edited pairs themselves, pairs sharing one end point with an edit, the pair whose end points both had an edit to
    the same third node, and hub-row pairs with the hub first and second."""
    n = A.shape[0]
    has = lambda i, j: A[i, j] != 0
    nbrs = lambda v: [int(x) for x in A.indices[A.indptr[v]:A.indptr[v + 1]] if x != v]
    pairs = list(tags["deleted"]) + list(tags["inserted"]) + list(tags["changed"]) + [tags["back"]]
    a, b, t = tags["third"]
    pairs += [(a, b), (b, a)]
    ends = sorted({v for p in pairs for v in p})
    for v in ends[::2]:
        nb = nbrs(v)
        if nb:
            pairs.append((v, nb[int(rng.integers(len(nb)))]))
        pairs.append((v, int(rng.integers(n))))
    for h in hubs:
        nb = np.array(nbrs(h))
        pairs += [(h, int(nb[nb < h].max())), (h, int(nb[nb > h].min()))]
        pairs += [(h, int(rng.integers(0, h))), (h, int(rng.integers(h + 1, n)))]
    seen, brk, mk = set(), [], []
    for i, j in pairs:
        if i == j or (i, j) in seen:
            continue
        seen.add((i, j))
        (brk if has(i, j) else mk).append((i + 1, j + 1))
    return np.array(brk, dtype=np.int64), np.array(mk, dtype=np.int64)


def _oracle_scores(O, A, E, b, tol, it=100):
    n = A.shape[0]
    out = np.zeros(len(E)), np.zeros(len(E), dtype=np.int64), np.zeros(len(E), dtype=bool)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        for h, (i, j) in enumerate(E):
            U, B = edge_UB(n, int(i), int(j), b)
            out[0][h], out[1][h], out[2][h] = O.trace_fun_update(A, U, B, tol, it, 0, "exp")
    return out


def _check_scores(res, ref, special, tol):
    x, itr, lk = res
    ox, oit, olk = ref
    assert np.array_equal(itr, oit), (itr, oit)
    assert np.array_equal(np.asarray(lk, dtype=bool), olk)
    err = np.abs(x - ox)
    assert np.all(err[~special] <= 1e-10 * np.maximum(np.abs(ox[~special]), 1e-3 * tol)), (err / np.abs(ox)).max()
    assert np.all(err[special] <= 1e-7 * np.maximum(np.abs(ox[special]), tol))


@pytest.fixture(scope="module")
def cand_cases(O, synth):
    cache = {}

    def get(gname):
        if gname in cache:
            return cache[gname]
        # both graphs scaled by a power of two to a spectral radius near 1: the scores are then far above the
        # roundoff of exp(A) itself (unscaled, oregon_A7's smaller updates sit at 1e-4 of exp(normest) and differ
        # from the oracle by 2e-10 relative on the unedited path too), and every value stays dyadic
        if gname == "synthetic":
            A0 = synth["valued"]
            calls, tags = edit_script(A0, synth["isolated"], synth["hubs"], 6, 0.125)
            hubs = synth["hubs"]
        else:
            A0 = load_graph(gname)
            deg = np.diff(A0.indptr)
            order = np.argsort(-deg, kind="stable")
            hubs = [int(v) for v in order[:3]]
            low = np.sort(order[::-1][:6])                   # stand-ins for isolated nodes: the lowest degrees
            calls, tags = edit_script(A0, low, hubs, 6, 1.0)
        s = _pow2_scale(O, A0)
        A0 = (A0 * s).tocsr()
        calls = [[(i, j, v * s) for i, j, v in c] for c in calls]
        b = 0.5
        A = apply_edits(A0, calls)
        brk, mk = _candidate_lists(A, tags, hubs, np.random.default_rng(7))
        assert 16 < len(brk) <= 148 and 16 < len(mk) <= 148, (len(brk), len(mk))   # slot re-seeding; one-CTA path
        nrm, _ = O.normest(A, 1e-2)
        tol = 1e-8 * float(np.exp(nrm))
        ref = dict(brk=_oracle_scores(O, A, brk, -b, tol), mk=_oracle_scores(O, A, mk, b, tol))
        loop = tags["third"][2]
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            U, B = edge_UB(A.shape[0], loop + 1, loop + 1, 1.0)
            ref["loop"] = O.trace_fun_update(A, U, B, tol, 100, 0, "exp")
        cache[gname] = dict(A0=A0, A=A, calls=calls, brk=brk, mk=mk, b=b, tol=tol, ref=ref, loop=loop)
        return cache[gname]
    return get


@pytest.mark.parametrize("pipeline", ["one_cta", "slots16"])
@pytest.mark.parametrize("gname", ["synthetic", "oregon_A7"])
def test_candidate_scores_after_edits(kr, cand_cases, monkeypatch, gname, pipeline):
    """kr_trace_fun_update_edges on a matrix with pending edits: pair_small_kernel (one CTA per candidate) and, with
    KR_PAIR_SLOTS=16, the batched pipeline whose pair_seed_kernel re-seeds slots.  Then a self-loop candidate, which
    folds the edits in first, and the same pairs again on the folded matrix."""
    c = cand_cases(gname)
    A, tol, b = c["A"], c["tol"], c["b"]
    if pipeline == "slots16":
        monkeypatch.setenv("KR_PAIR_SLOTS", "16")
    M = kr.Matrix(c["A0"])
    for call in c["calls"]:
        assert set_edges(M, call) <= delta_bytes_bound(4 * len(call) + 64, A.shape[0])
    sb, sm = _special(A, c["brk"]), _special(A, c["mk"])
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        _check_scores(kr.trace_fun_update_edges(M, c["brk"], -b, tol, 100, "exp"), c["ref"]["brk"], sb, tol)
        _check_scores(kr.trace_fun_update_edges(M, c["mk"], b, tol, 100, "exp"), c["ref"]["mk"], sm, tol)
        loop = np.array([[c["loop"] + 1, c["loop"] + 1]], dtype=np.int64)
        x, itr, lk = kr.trace_fun_update_edges(M, loop, b, tol, 100, "exp", b_self=1.0)
        ox, oit, olk = c["ref"]["loop"]
        assert itr[0] == oit and bool(lk[0]) == bool(olk) and abs(x[0] - ox) <= 1e-10 * abs(ox)
        _check_scores(kr.trace_fun_update_edges(M, c["brk"], -b, tol, 100, "exp"), c["ref"]["brk"], sb, tol)
        _check_scores(kr.trace_fun_update_edges(M, c["mk"], b, tol, 100, "exp"), c["ref"]["mk"], sm, tol)
    assert_spmm_exact(kr, M, A, 60, ks=(5,))


# ------------------------------------------------------------------ 6. the node screen
@pytest.mark.parametrize("pipeline", ["one_cta", "slots16"])
def test_screened_round_after_edits(kr, O, synth, monkeypatch, pipeline):
    """kr_greedy_round with the node screen on a matrix with pending edits among the candidates' nodes: the same
    winner and value as an exact round on the edited matrix built afresh, the contenders re-scored through
    pair_small_kernel or (KR_PAIR_SLOTS=16) the batched pipeline."""
    A0 = synth["pattern"]
    s = _pow2_scale(O, A0)
    A0 = (A0 * s).tocsr()
    c = O.compute_centrality(A0, "eig")
    E = np.asarray(kr.find_top_missing_edges(A0, c, 600, "min"), dtype=np.int64)
    nodes = np.unique(E) - 1
    assert len(E) >= 8 * nodes.size and A0.shape[0] > 130         # node_screen_applicable
    rng = np.random.default_rng(11)
    call = [(int(E[h, 0]) - 1, int(E[h, 1]) - 1, 0.5 * s) for h in rng.choice(len(E), 4, replace=False)]
    sub = sp.triu(A0[nodes][:, nodes], 1).tocoo()
    pick = rng.choice(sub.nnz, 5, replace=False)
    call += [(int(nodes[sub.row[q]]), int(nodes[sub.col[q]]), 0.0) for q in pick[:3]]
    call += [(int(nodes[sub.row[q]]), int(nodes[sub.col[q]]), -1.25 * s) for q in pick[3:]]
    A = apply_edits(A0, [call])
    nrm, _ = O.normest(A, 1e-2)
    tol = 1e-8 * float(np.exp(nrm))
    b0, v0, _, _, _ = kr.greedy_round(kr.Matrix(A), E, s, tol, 100, "exp", "make", screen=False)
    if pipeline == "slots16":
        monkeypatch.setenv("KR_PAIR_SLOTS", "16")
    M = kr.Matrix(A0)
    set_edges(M, call)
    b1, v1, scores, mask, info = kr.greedy_round(M, E, s, tol, 100, "exp", "make", screen=True)
    assert info["screened"] > 0, info
    assert b1 == b0 and abs(v1 - v0) <= 1e-10 * abs(v0), (b1, b0, v1, v0)
    top = np.where(mask)[0][np.argsort(-scores[mask])[:3]]
    ref = _oracle_scores(O, A, E[top], s, tol)
    _check_scores((scores[top], ref[1], ref[2]), ref, _special(A, E[top]), tol)
    assert_spmm_exact(kr, M, A, 70, ks=(5,))


# ------------------------------------------------------------------ 7. unsymmetric matrices
def test_unsymmetric_edits_rebuild_the_transpose(kr, O):
    rng = np.random.default_rng(8)
    n = 3000
    S = sp.random(n, n, density=0.003, random_state=8, data_rvs=lambda k: rng.integers(1, 17, k) / 8.0)
    S = sp.triu(S, 1)
    L = (S + S.T).tolil()
    asym = []
    for i, j in rng.choice(n, (12, 2), replace=False):
        L[i, j] = 1.5
        L[j, i] = 0.0 if len(asym) % 3 == 0 else -0.25
        asym.append((int(i), int(j)))
    A0 = L.tocsr()
    A0.eliminate_zeros()
    assert abs(A0 - A0.T).nnz > 0
    M = kr.Matrix(A0)
    assert not M.info()["symmetric"]
    # symmetrise half the unsymmetric pairs, insert and delete elsewhere: still unsymmetric, rebuilt with its transpose
    T = sp.triu(A0, 1).tocoo()
    call1 = [(i, j, 0.75) for i, j in asym[:6]] + [(int(T.row[q]), int(T.col[q]), 0.0) for q in range(5)]
    call1 += [(int(a), int(b), -0.5) for a, b in rng.integers(0, n, (5, 2))]
    shipped = set_edges(M, call1)
    A1 = apply_edits(A0, [call1])
    assert shipped >= 4 * A1.nnz
    _info_matches(M, A1)
    assert_spmm_exact(kr, M, A1, 80, ks=(1, 17))
    e, cnt = kr.normest(M, 1e-6)
    oe, ocnt = O.normest(A1, 1e-6)
    assert cnt == ocnt and abs(e - oe) <= 1e-12 * oe
    for p in (2, 5):
        c, mv = kr.normAm(M, p)
        oc, omv = O.normAm(A1, p)
        assert mv == omv and abs(c - oc) <= 1e-12 * oc
    bvec = rng.standard_normal((n, 3))
    for t in (1.0, -0.5):
        f, s_, m, mv, mvd, unA = kr.expmv(t, M, bvec, None, "double", True, False, False)
        of, os_, om, omv, omvd, ounA = O.expmv(t, A1, bvec, None, "double", True, False, False)
        assert [s_, m, mv, mvd, unA] == [os_, om, omv, omvd, ounA]
        assert np.max(np.abs(f - of)) <= 1e-10 * np.max(np.abs(of))
    # the other half: symmetric again, and later edits take the delta path
    call2 = [(j, i, 0.75) for i, j in asym[6:]]
    set_edges(M, call2)
    A2 = apply_edits(A1, [call2])
    assert abs(A2 - A2.T).nnz == 0
    assert _info_matches(M, A2)["symmetric"]
    assert_spmm_exact(kr, M, A2, 90, ks=(5,))
    call3 = [(int(a), int(b), 1.25) for a, b in rng.integers(0, n, (4, 2))]
    assert set_edges(M, call3) <= delta_bytes_bound(8, n)
    A3 = apply_edits(A2, [call3])
    assert_spmm_exact(kr, M, A3, 95, ks=(5,))
    c, mv = kr.normAm(M, 3)
    oc, omv = O.normAm(A3, 3)
    assert mv == omv and abs(c - oc) <= 1e-12 * oc


# ------------------------------------------------------------------ 8. kr_matrix_info
@pytest.mark.parametrize("variant", ["pattern", "valued"])
def test_info_describes_the_edited_matrix(kr, O, synth, variant):
    """nnz, nonnegative and symmetric of the edited matrix while the edits are pending, without folding them in
    (nothing is uploaded and the SpMM still applies the deltas), and after a fold.  pattern_only describes the
    storage."""
    A0 = synth[variant]
    unit = 0.25 if variant == "pattern" else 0.125
    calls, _ = edit_script(A0, synth["isolated"], synth["hubs"], 12, unit)
    M = kr.Matrix(A0)
    for step, call in enumerate(calls):
        set_edges(M, call)
        A = apply_edits(A0, calls[:step + 1])
        before = M.ctx.counters()
        info = _info_matches(M, A)
        assert M.ctx.counters() == before
        assert info["pattern_only"] == (variant == "pattern")
        assert_spmm_exact(kr, M, A, 110 + step, ks=(5,))
    assert A.nnz != A0.nnz and not np.all(A.data >= 0)
    kr.normest(M, 1e-2)                                               # folds the edits in
    info = _info_matches(M, A)
    assert info["pattern_only"] == bool(np.all(A.data == A.data[0]))


def test_info_nonnegative_follows_the_edits(kr):
    """A stored negative entry cleared by an edit, a new negative value, and its removal."""
    rng = np.random.default_rng(13)
    n = 500
    S = sp.triu(sp.random(n, n, density=0.02, random_state=13, data_rvs=lambda k: rng.integers(1, 9, k) / 4.0), 1)
    S = S.tolil()
    S[3, 70] = -0.5
    S[10, 200] = -1.0
    A = (S + S.T).tocsr()
    M = kr.Matrix(A)
    assert not M.info()["nonnegative"]
    steps = [[(3, 70, 0.25)], [(200, 10, 0.0)], [(5, 6, -2.0), (7, 7, 1.0)], [(6, 5, 0.5)], [(7, 7, -0.25)],
             [(7, 7, 0.0)], [(70, 3, -0.5)]]
    expect = [False, True, False, True, False, True, False]
    for k, (call, nonneg) in enumerate(zip(steps, expect)):
        set_edges(M, call)
        Ak = apply_edits(A, steps[:k + 1])
        assert _info_matches(M, Ak)["nonnegative"] == nonneg, k
        assert_spmm_exact(kr, M, Ak, 120 + k, ks=(3,))
