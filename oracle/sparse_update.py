"""tr f(Ã) - tr f(Ã - D) for a sparse symmetric direction D = Δ(X, Ω): the method of kr_trace_fun_sparse_update
(csrc/sparse_update.cuh), restated over this package's function_multiple_entries.

D has D(i,j) = D(j,i) = X_h for every row (i, j) of Ω (duplicates add up; a diagonal pair gives D(i,i) = X_h).  With
A_t = Ã - (1 - t) D, so that A_0 = Ã - D and A_1 = Ã,

    tr f(Ã) - tr f(A_0) = ∫₀¹ φ'(t) dt,   φ(t) = tr f(A_t),   φ'(t) = tr(f'(A_t) D) = Σ_h c_h X_h f'(A_t)(i_h, j_h)

with c_h = 2 off the diagonal and 1 on it, f' = exp / cosh / sinh for f = exp / sinh / cosh.  The integral is taken by
q-point Gauss-Legendre on [0, 1], whose error is (q!)^4 / ((2q+1) ((2q)!)^3) φ^(2q)(ξ) for some ξ in [0, 1].

The bound on φ^(2q).  Write f(x) = Σ_k a_k x^k; for exp, sinh and cosh |a_k| <= 1/k!.  A_t = A_0 + tD, so the m-th
derivative of tr (A_0 + tD)^k is m! times the sum over the C(k, m) words with m letters D and k - m letters A_t, i.e.
k!/(k-m)! words, each of trace at most n ||D||^m ||A_t||^(k-m) (|tr M| <= n ||M|| for any n x n M, and the norm of a
word is at most the product of its letters' norms).  With r = ||A_t|| <= ||Ã|| + (1 - t) ||D|| <= ||Ã|| + ||D|| =: ρ,

    |φ^(m)(t)| <= n Σ_{k>=m} (1/k!) k!/(k-m)! ||D||^m r^(k-m) = n ||D||^m e^r <= n ||D||^m e^ρ.

q is the smallest order with (q!)^4 / ((2q+1) ((2q)!)^3) n ||D||^{2q} e^ρ <= tol Σ_h c_h |X_h| - the error the entries'
own stopping tolerance already allows in the sum - with ||D|| bounded by its infinity norm and ||Ã|| taken from
normest; at most min(qmax, 32).  tests/test_oracle_sparse_update.py checks the bound against the quadrature error.
"""
import math

import numpy as np
import scipy.sparse as sp

from .updates import fun_name, function_multiple_entries, normest

QCAP = 32
DERIV = {"exp": "exp", "sinh": "cosh", "cosh": "sinh"}


def delta(X, Omega, n):
    """D = Δ(X, Ω) as a CSR matrix (1-based Ω, duplicates summed, a diagonal pair counted once)."""
    Om = np.asarray(Omega, dtype=np.int64).reshape(-1, 2)
    X = np.asarray(X, dtype=np.float64).ravel()
    off = Om[:, 0] != Om[:, 1]
    r = np.concatenate([Om[:, 0], Om[off, 1]]) - 1
    c = np.concatenate([Om[:, 1], Om[off, 0]]) - 1
    return sp.csr_matrix((np.concatenate([X, X[off]]), (r, c)), shape=(n, n))


def log_error_bound(q, n, normD, normA):
    """log of (q!)^4 / ((2q+1) ((2q)!)^3) * n * ||D||^{2q} * e^{||A|| + ||D||}."""
    lD = math.log(normD) if normD > 0 else -math.inf
    return (4 * math.lgamma(q + 1) - math.log(2 * q + 1) - 3 * math.lgamma(2 * q + 1) + math.log(n) + 2 * q * lD
            + normA + normD)


def choose_q(n, normD, normA, tol, sumw, qmax=QCAP):
    qcap = min(int(qmax), QCAP)
    target = math.log(tol * sumw) if tol * sumw > 0 else -math.inf
    for q in range(1, qcap):
        if log_error_bound(q, n, normD, normA) <= target:
            return q
    return qcap


def gauss_legendre01(q):
    x, w = np.polynomial.legendre.leggauss(q)
    return 0.5 * (1.0 + x), 0.5 * w


def trace_fun_sparse_update(At, X, Omega, fun, tol, it=None, qmax=QCAP):
    """(dtr, q, iter): dtr = tr f(At) - tr f(At - D), D = delta(X, Omega); iter = the largest iteration count of the
    entries at any quadrature node.  X = 0 gives (0.0, 0, 0)."""
    At = sp.csr_matrix(At, dtype=np.float64)
    n = At.shape[0]
    if qmax < 1:
        raise ValueError("qmax must be >= 1")
    name = fun_name(fun)
    Om = np.asarray(Omega, dtype=np.int64).reshape(-1, 2)
    X = np.asarray(X, dtype=np.float64).ravel()
    keep = X != 0
    if not keep.any():
        return 0.0, 0, 0
    Om, X = Om[keep], X[keep]
    cx = np.where(Om[:, 0] == Om[:, 1], 1.0, 2.0) * X
    D = delta(X, Om, n)
    normD = float(abs(D).sum(axis=1).max())
    normA = float(normest(At, 1e-2)[0])
    q = choose_q(n, normD, normA, tol, float(np.abs(cx).sum()), qmax)
    t, w = gauss_legendre01(q)
    dtr, it_max = 0.0, 0
    for tq, wq in zip(t, w):
        vals, itq = function_multiple_entries((At - (1.0 - tq) * D).tocsr(), Om, DERIV[name], tol, it)
        dtr += wq * float(np.dot(cx, vals))
        it_max = max(it_max, int(itq))
    return dtr, q, it_max
