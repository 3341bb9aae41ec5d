"""Oracle: edge scores with a value per candidate, and the weighted greedy driver.  TEST INFRASTRUCTURE ONLY.

The candidate loop of functions/krylov_miobi.m:76-99 with B = d_h [0 1; 1 0] per candidate (the reference has one value,
sign / rescale, for all of them) - each candidate through the existing oracle trace_fun_update
(functions/trace_fun_update.m) - and greedy_krylov (functions/greedy_krylov.m) with the edits that were scored: a removed
edge loses its stored weight, an inserted one gets its own weight.
"""
import warnings

import numpy as np
import scipy.sparse as sp

from .greedy import _issymmetric, _set_edge, find_top_edges, find_top_missing_edges
from .updates import trace_fun_update


def trace_fun_update_edges_w(A, E, d, tol=1e-12, it=None, fun="exp"):
    """(Xm, iter, lucky) arrays: row h = (i, j) of E (1-based) scored with U = [e_i e_j], B = d[h] [0 1; 1 0]; a self
    loop i == j with U = e_i, B = d[h]."""
    A = sp.csr_matrix(A).astype(np.float64)
    n = A.shape[0]
    E = np.atleast_2d(np.asarray(E)).astype(np.int64)
    d = np.broadcast_to(np.asarray(d, dtype=np.float64), (E.shape[0],))
    x = np.zeros(E.shape[0])
    its = np.zeros(E.shape[0], dtype=np.int64)
    lucky = np.zeros(E.shape[0], dtype=bool)
    for h, (i, j) in enumerate(E):
        if i != j:
            U = np.zeros((n, 2))
            U[i - 1, 0] = 1.0
            U[j - 1, 1] = 1.0
            B = d[h] * np.array([[0.0, 1.0], [1.0, 0.0]])
        else:
            U = np.zeros((n, 1))
            U[i - 1, 0] = 1.0
            B = np.array([[d[h]]])
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            x[h], its[h], lucky[h] = trace_fun_update(A, U, B, tol, it, 0, fun)
    return x, its, lucky


def greedy_krylov_weighted(A, k, Q=0, centrality=None, order="mult", tol=1e-12, it=None, fun="exp", miobi="break",
                           weights=None):
    """(edges, rob_variation, A_new, applied): greedy_krylov.m:1-97 with per-candidate values.  'break': candidates
    find_top_edges(A, centrality, Q + k, order), d_h = -A(i_h, j_h) of the current A, the chosen edge set to 0.  'make':
    candidates find_top_missing_edges(A, centrality, Q + k, order), d_h = +w_h (weights: scalar or aligned with that
    list, default 1), the chosen pair set to w_h.  Selection: krylov_miobi.m:112-124 (strict compare, first wins)."""
    if not _issymmetric(A):
        raise ValueError("GREEDY_KRYLOV:: Adjacency matrix should be symmetric")
    A = sp.csr_matrix(A).astype(np.float64)
    if it is None:
        it = min(100, A.shape[0])
    if not Q:
        Q = int(np.asarray(A.sum(axis=0)).max())
    top = (find_top_missing_edges if miobi == "make" else find_top_edges)(A, centrality, Q + k, order)
    w = None
    if miobi == "make":
        w = np.array(np.broadcast_to(np.asarray(1.0 if weights is None else weights, dtype=np.float64), (top.shape[0],)))
    rob, edges, applied, chosen = 0.0, np.zeros((0, 2), dtype=np.int64), [], None
    for j in range(1, min(k, top.shape[0]) + 1):
        if j > 1:                                           # greedy_krylov.m:84-86
            keep = ~np.all(top == chosen, axis=1)
            top = top[keep]
            w = w[keep] if w is not None else None
        E = top[:Q]
        d = w[:E.shape[0]] if w is not None else -np.array([A[a - 1, b - 1] for a, b in E])
        vals = trace_fun_update_edges_w(A, E, d, tol, it, fun)[0]
        best, bestval = -1, (np.inf if miobi == "break" else -np.inf)
        for h in range(E.shape[0]):                         # krylov_miobi.m:112-124
            if (miobi == "break" and vals[h] < bestval) or (miobi == "make" and vals[h] > bestval):
                best, bestval = h, vals[h]
        chosen = E[best].copy()
        A = _set_edge(A, int(chosen[0]), int(chosen[1]), 0.0 if miobi == "break" else float(d[best]))
        edges = np.vstack([edges, chosen[None, :]])
        rob += bestval
        applied.append(float(d[best]))
    return edges, rob, A, np.asarray(applied)
