"""Oracle: node removal scored by the Krylov path, and the greedy node attack.  TEST INFRASTRUCTURE ONLY.

Removing node v is the rank-two update U = [e_v, a'], B = -[0 1; 1 0] of trace_fun_update.m:72-124 (a' the
off-diagonal part of row v).  range(U) lies in K_2(A, e_v), so K_j(A, U) = K_{j+1}(A, e_v): the projected update is a
single-vector Lanczos run from e_v, restated here with the three-term recurrence the device path runs.
"""
import numpy as np
import scipy.sparse as sp

from .greedy import _issymmetric, compute_centrality
from .updates import _trace_formula, fun_name


def lanczos_three_term(A, v, steps):
    """alpha_1..alpha_steps, beta_1..beta_steps of the single-vector Lanczos run from e_v (0-based v): the recurrence of
    lanczos_krylov.m:73-101 with bs = 1, but with the three-term update in place of CGS2 against the window (the device
    path of kr_trace_fun_update_nodes runs this one, so iteration counts agree).  The basis is kept unnormalised,
    v_j = s_j u_j, exactly as the device keeps it: beta = 0 leaves a zero vector with scale 0 (no NaN)."""
    n = A.shape[0]
    u1 = np.zeros(n)
    u1[v] = 1.0
    u0 = np.zeros(n)
    s1, s0, bprev = 1.0, 0.0, 0.0
    alpha, beta = np.zeros(steps), np.zeros(steps)
    for i in range(steps):
        y = np.asarray(A @ u1).ravel()
        a = s1 * s1 * float(u1 @ y)
        w = s1 * y + (-a * s1) * u1 + (-bprev * s0) * u0
        b = float(np.sqrt(w @ w))
        alpha[i], beta[i] = a, b
        s0, s1, bprev = s1, (1.0 / b if b > 0.0 else 0.0), b
        u0, u1 = u1, w
    return alpha, beta


def trace_fun_update_node(A, v, tol=1e-12, it=None, fun="exp"):
    """[Xm, iter, lucky] for the removal of node v (1-based): tr f(Ã) - tr f(A), Ã = A with the off-diagonal entries of
    row and column v set to zero (a_vv kept).  trace_fun_update.m:72-124 with U = [e_v, a'] (a' the off-diagonal part of
    row v), B = -[0 1; 1 0], restated on K_j(A, U) = K_{j+1}(A, e_v): at step j Gm = T_{j+1}, tGm = Gm with its (1,2)
    and (2,1) entries zeroed; lag-2 rule (:104-118), then the lucky exit (:119-124, beta_{j+1} < 1e-8).  A node without
    off-diagonal entries scores 0 with iter 1, lucky."""
    name = fun_name(fun)
    A = sp.csr_matrix(A)
    n = A.shape[0]
    if it is None:
        it = min(100, n)
    alpha, beta = lanczos_three_term(A, int(v) - 1, it + 1)
    if not beta[0] >= 1e-8:
        return 0.0, 1, True
    Xstop = [0.0, 0.0]
    Xm, lucky, j = 0.0, False, 0
    for j in range(1, it + 1):
        N = j + 1
        Gm = np.diag(alpha[:N]) + np.diag(beta[:N - 1], 1) + np.diag(beta[:N - 1], -1)
        tGm = Gm.copy()
        tGm[0, 1] = tGm[1, 0] = 0.0
        Xm = _trace_formula(name, np.linalg.eigvalsh(tGm), np.linalg.eigvalsh(Gm))
        lucky = not beta[j] >= 1e-8
        if j <= 2:
            Xstop[j - 1] = Xm
        elif abs(Xm - Xstop[0]) < tol:
            break
        else:
            Xstop = Xstop[1:] + [Xm]
        if lucky:
            break
    return Xm, j, bool(lucky)


def _remove_node(A, v):
    """A with the off-diagonal entries of row and column v (1-based) deleted; a_vv stays."""
    A = A.tolil()
    for j in A.rows[v - 1][:]:
        if j != v - 1:
            A[v - 1, j] = 0.0
            A[j, v - 1] = 0.0
    A = A.tocsr()
    A.eliminate_zeros()
    return A


def greedy_krylov_nodes(A, k, Q=0, centrality=None, tol=1e-12, it=None, fun="exp"):
    """[nodes, rob_variation, A_new]: greedy node attack, the node counterpart of greedy_krylov.m:1-97.  Round 1 ranks
    the nodes by centrality (descending, stable) and keeps the top Q + k; every round scores the first Q remaining
    nodes by trace_fun_update_node, takes the first-wins arg-min (krylov_miobi.m:112-124), deletes the chosen node's
    off-diagonal entries and drops it from the list.  Q = 0 takes the reference's default, max column sum of A.
    centrality = None: 'eig' centrality."""
    if not _issymmetric(A):
        raise ValueError("GREEDY_KRYLOV:: Adjacency matrix should be symmetric")
    A = sp.csr_matrix(A).astype(np.float64)
    n = A.shape[0]
    if it is None:
        it = min(100, n)
    if not Q:
        Q = int(np.asarray(A.sum(axis=0)).max())
    if centrality is None:
        centrality = compute_centrality(A, "eig")
    top = np.argsort(-np.asarray(centrality, dtype=np.float64).ravel(), kind="stable")[:Q + k] + 1
    nodes, rob_variation = [], 0.0
    for _ in range(min(k, top.size)):
        cand = top[:Q]
        vals = np.array([trace_fun_update_node(A, v, tol, it, fun)[0] for v in cand])
        best, bestval = -1, np.inf
        for h in range(cand.size):
            if vals[h] < bestval:
                best, bestval = h, vals[h]
        chosen = int(cand[best])
        A = _remove_node(A, chosen)
        top = top[top != chosen]
        nodes.append(chosen)
        rob_variation += bestval
    return np.asarray(nodes, dtype=np.int64), rob_variation, A
