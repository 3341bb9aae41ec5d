"""Oracle: the Hessian of the all-edges callbacks times vectors, per row over multiple_frechet_eval.  TEST
INFRASTRUCTURE ONLY.

For every pair h = (i, j) of Omega, multiple_frechet_eval (functions/multiple_frechet_eval.m) gives the Arnoldi bases
U of K_s(Atilde, e_i) and V of K_s(Atilde, e_j) and X_h, the (1,2) block of f([G, e1 e1'; 0, H']) at the pair's stop
step s.  Then
    W(h, r) = -2 <X_h, U' S_r V>_F,   S_r = sum_l Y(l, r) e_a e_b'  (+ e_b e_a' in the objective form), (a, b) = Omega(l, :).
The reference form is hessianfcn_fun's Hes * Y (functions/hessianfcn_fun.m:8-15) with every row from its own X_h;
the objective form is the Hessian of -(tr fun(Atilde) - tr fun(A)), whose X-derivative of Atilde is e_a e_b' + e_b e_a'.
"""
import numpy as np
import scipy.sparse as sp

from .frechet import multiple_frechet_eval


def direction(Y, Omega, n, reference_form):
    """S_r for every column r of Y (len(Omega) x p): list of n x n CSR matrices (duplicates add up)."""
    Om = np.atleast_2d(np.asarray(Omega)).astype(np.int64)
    out = []
    for y in Y.T:
        S = sp.csr_matrix((y, (Om[:, 0] - 1, Om[:, 1] - 1)), shape=(n, n))
        out.append(S if reference_form else (S + S.T).tocsr())
    return out


def hessian_multiply(X, A, Omega, f, Y, tol, it, reference_form=False, rows=None):
    """(W, iter): W = Hes * Y on Atilde = A + Delta(X, Omega) (hessianfcn_fun.m:4-7), Y of shape len(Omega) or
    len(Omega) x p.  rows evaluates a subset of the pairs (W then has len(rows) rows); a pair's X_h and bases do not
    depend on the other pairs, so the subset gives the same rows.  iter is multiple_frechet_eval's step count."""
    n = A.shape[0]
    Om = np.atleast_2d(np.asarray(Omega)).astype(np.int64)
    X = np.asarray(X, dtype=np.float64).ravel()
    XX = sp.csr_matrix((X, (Om[:, 0] - 1, Om[:, 1] - 1)), shape=(n, n))
    At = (sp.csr_matrix(A) + XX + XX.T).tocsr()
    Y = np.asarray(Y, dtype=np.float64)
    vec = Y.ndim == 1
    Yc = Y.reshape(len(Om), -1)
    sub = Om if rows is None else Om[np.asarray(rows, dtype=np.int64)]
    Um, Xm, Vm, row, col, itu = multiple_frechet_eval(At, sub, f, tol, it)
    Ss = direction(Yc, Om, n, reference_form)
    W = np.zeros((len(sub), Yc.shape[1]))
    for h, (i, j) in enumerate(sub):
        s0, s1 = Xm[h].shape
        U = Um[row[int(i)]][:, :s0]
        V = Vm[col[int(j)]][:, :s1]
        for r, S in enumerate(Ss):
            W[h, r] = -2.0 * np.sum(Xm[h] * (U.T @ (S @ V)))
    return (W[:, 0] if vec else W), itu
