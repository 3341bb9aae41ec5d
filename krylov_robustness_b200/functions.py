"""Host-side mirror of the reference's function interface (functions/*.m), same names, argument
order, defaults and error strings - each a thin marshaller into the C ABI of libkrylov_b200.so.

``A`` may be a SciPy sparse matrix / dense array (uploaded on each call) or an ``engine.Matrix``
(device-resident, the analogue of passing the operator struct of lanczos_krylov.m:78-79).
Index lists are 1-based as in the reference.  Function selectors are 'exp' / 'sinh' / 'cosh'
(or np.exp / np.sinh / np.cosh).  No function here computes on the CPU.
"""
import ctypes as C
import math
import warnings

import numpy as np
import scipy.sparse as sp

from ._lib import check
from .engine import Context, Matrix, Dense, fun_id, _ptr, _f64_cm


__all__ = ["slq_trace", "lanczos_krylov", "arnoldi_krylov", "trace_fun_update", "trace_fun_update_edges",
           "fun_update", "function_multiple_entries", "fun_and_grad_krylov_exp", "fun_and_grad_krylov_fun",
           "normest", "normAm", "select_taylor_degree", "expmv", "ExpmvHandle", "mc_trace", "trace_exp",
           "edge2low_rank", "compute_centrality", "find_top_edges", "find_top_missing_edges",
           "select_candidate", "greedy_round", "krylov_miobi", "greedy_krylov", "trace_fun_update_nodes", "greedy_krylov_nodes",
           "trace_fun_sparse_update", "KrylovParams", "fun_and_grad_all_edges", "hessp_all_edges", "hessianfcn_exp",
           "hessianfcn_fun"]


def _mat(A, ctx=None):
    return Matrix.wrap(A, ctx)


# ----------------------------------------------------------------------------- throughput mode
def slq_trace(A, Z, m=30, fun="exp", return_details=False):
    """Throughput-mode estimator (SURVEY.md 8d, C3): mean_z ||z||^2 e1' f(T_z) e1 over all probe
    columns of Z at once.  Z: n x k array (host) or engine.Dense (device-resident)."""
    M = _mat(A)
    lib, ctx = M.ctx.lib, M.ctx
    tr = C.c_double()
    sign = False
    if isinstance(Z, Dense):
        k = Z.k
    elif isinstance(Z, np.ndarray) and Z.dtype == np.int8:
        # Rademacher probes as int8 signs: 1/8 of the upload, expanded to fp64 on the device
        sign = True
        Z = Z if Z.ndim == 2 else Z[:, None]
        if not (Z.strides[0] == 1 and Z.strides[1] >= max(Z.shape[0], 1)):      # column-major with any ld is taken as is
            Z = np.asfortranarray(Z)
        ldz, k = (Z.strides[1] if Z.shape[1] > 1 else max(Z.shape[0], 1)), Z.shape[1]
    else:
        Z, ldz = _f64_cm(Z)
        k = Z.shape[1]
    vals = np.empty(k) if return_details else None
    al = np.empty((m, k), order="F") if return_details else None
    be = np.empty((m, k), order="F") if return_details else None
    if isinstance(Z, Dense):
        check(lib.kr_slq_trace_dev(ctx.h, M.h, Z.h, m, fun_id(fun), C.byref(tr), _ptr(vals), _ptr(al), _ptr(be)))
    else:
        entry = lib.kr_slq_trace_sign if sign else lib.kr_slq_trace
        check(entry(ctx.h, M.h, k, _ptr(Z), ldz, m, fun_id(fun), C.byref(tr), _ptr(vals), _ptr(al), _ptr(be)))
    if return_details:
        return tr.value, vals, al, be
    return tr.value


def _default_it(M, it):
    return int(min(100, M.n)) if it is None else int(it)


def _is_exp(fun):
    return fun_id(fun) == 0


# ----------------------------------------------------------------------------- L1: basis builders
class KrylovParams:
    """The reference's ``params`` struct (functions/lanczos_krylov.m:55-57).  ``last`` / ``A`` are
    kept for interface parity; the live state is the device handle."""

    def __init__(self, M, handle, arnoldi):
        self.A = M
        self._h = handle
        self._arnoldi = arnoldi
        self._lib = M.ctx.lib

    @property
    def last(self):
        return self._fetch()[3]

    def _dims(self):
        d = (C.c_int64 * 5)()
        check(self._lib.kr_krylov_dims(self._h, d))
        return list(d)

    def _fetch(self):
        bs, steps, hr, hc, vc = self._dims()
        n = self.A.n
        V = np.empty((n, vc), order="F")
        H = np.empty((hr, hc), order="F")
        K = np.zeros((hr, hc), order="F") if self._arnoldi else None
        last = np.empty((n, bs), order="F")
        check(self._lib.kr_krylov_get(self._h, _ptr(V), max(n, 1), _ptr(H), max(hr, 1), _ptr(K), max(hr, 1),
                                      _ptr(last), max(n, 1)))
        return V, H, K, last

    def __del__(self):
        try:
            if self._h:
                self._lib.kr_krylov_destroy(self._h)
                self._h = None
        except Exception:
            pass


def _krylov(args, arnoldi):
    nstart, next_ = (2, 4) if arnoldi else (2, 3)
    if len(args) not in (nstart, next_):
        raise ValueError("Called with the wrong number of arguments")
    lucky = C.c_int()
    if len(args) == 2:
        A, b = args
        M = _mat(A)
        b, ldb = _f64_cm(b)
        if b.shape[0] != M.n:
            raise ValueError("The block vector b has wrong number of rows")
        h = C.c_void_p()
        check(M.ctx.lib.kr_krylov_start(M.ctx.h, M.h, int(arnoldi), b.shape[1], _ptr(b), ldb, C.byref(h),
                                        C.byref(lucky)))
        params = KrylovParams(M, h, arnoldi)
    else:
        params = args[-1]
        check(params._lib.kr_krylov_extend(params._h, C.byref(lucky)))
    V, H, K, _ = params._fetch()
    if arnoldi:
        return V, K, H, params, bool(lucky.value)
    return V, H, params, bool(lucky.value)


def lanczos_krylov(*args):
    """[V,H,params,lucky] = lanczos_krylov(A,b) | lanczos_krylov(V,H,params)
    (functions/lanczos_krylov.m:1-67).  V is the retained two-block window, H block tridiagonal."""
    return _krylov(args, False)


def arnoldi_krylov(*args):
    """[V,K,H,params,lucky] = arnoldi_krylov(A,b) | arnoldi_krylov(V,K,H,params)
    (functions/arnoldi_krylov.m:1-72)."""
    return _krylov(args, True)


# ----------------------------------------------------------------------------- L2: evaluators
def trace_fun_update(A, U, B, tol=1e-12, it=None, debug=0, fun="exp"):
    """[Xm,iter,lucky] = trace_fun_update(A,U,B,tol,it,debug,fun)  (functions/trace_fun_update.m:1-130)."""
    M = _mat(A)
    it = _default_it(M, it)
    if sp.issparse(U):
        U = U.toarray()
    U, ldu = _f64_cm(U)
    if U.shape[0] != M.n:
        raise ValueError("The block vector b has wrong number of rows")
    B, ldb = _f64_cm(np.atleast_2d(np.asarray(B, dtype=np.float64)))
    x, k, lucky = C.c_double(), C.c_int64(), C.c_int()
    check(M.ctx.lib.kr_trace_fun_update(M.ctx.h, M.h, U.shape[1], _ptr(U), ldu, _ptr(B), ldb, float(tol), it,
                                        fun_id(fun), C.byref(x), C.byref(k), C.byref(lucky)))
    if k.value == it:
        warnings.warn("TRACE_FUN_UPDATE:: Reached maximum number of iterations")
    return x.value, k.value, bool(lucky.value)


def trace_fun_update_edges(A, E, b_offdiag, tol=1e-12, it=None, fun="exp", b_self=None):
    """All candidates of the loop at functions/krylov_miobi.m:76-99 in one call: for each row (i, j) of
    E (1-based) U = [e_i e_j], B = b_offdiag*[0 1;1 0]; a self loop i == j is the rank-one update B = b_self
    (default b_offdiag; the reference does not rescale it, krylov_miobi.m:88-94).
    Returns (Xm, iter, lucky) arrays."""
    M = _mat(A)
    it = _default_it(M, it)
    E = np.asfortranarray(np.atleast_2d(np.asarray(E)).astype(np.int64))
    nE = E.shape[0]
    x = np.zeros(nE)
    k = np.zeros(nE, dtype=np.int64)
    lucky = np.zeros(nE, dtype=np.int32)
    check(M.ctx.lib.kr_trace_fun_update_edges_ex(M.ctx.h, M.h, nE, _ptr(E), float(b_offdiag),
                                                 float(b_offdiag if b_self is None else b_self), float(tol), it,
                                                 fun_id(fun), _ptr(x), _ptr(k), _ptr(lucky)))
    return x, k, lucky.astype(bool)


def trace_fun_update_nodes(A, nodes, tol=1e-12, it=None, fun="exp"):
    """Node-removal scores, all candidates in one call (kr_trace_fun_update_nodes): for every node v (1-based)
    tr f(Ã) - tr f(A), Ã = A with the off-diagonal entries of row and column v set to zero (a_vv kept).  The
    reference's trace_fun_update (functions/trace_fun_update.m:72-124) with U = [e_v, a'], B = -[0 1; 1 0], run as a
    single-vector Lanczos from e_v; same lag-2 and lucky-breakdown stops.  Returns (Xm, iter, lucky) arrays."""
    M = _mat(A)
    it = _default_it(M, it)
    V = np.ascontiguousarray(np.asarray(nodes).ravel(), dtype=np.int64)
    x = np.zeros(V.size)
    k = np.zeros(V.size, dtype=np.int64)
    lucky = np.zeros(V.size, dtype=np.int32)
    check(M.ctx.lib.kr_trace_fun_update_nodes(M.ctx.h, M.h, V.size, _ptr(V), float(tol), it, fun_id(fun), _ptr(x),
                                              _ptr(k), _ptr(lucky)))
    return x, k, lucky.astype(bool)


def greedy_round(A, E, b_offdiag, tol=1e-12, it=None, fun="exp", miobi="break", screen=True, b_self=None):
    """One round of the greedy loop (functions/krylov_miobi.m:76-124): score the candidates E and select arg-min
    ('break') / arg-max ('make') with the reference's strict first-wins rule - kr_greedy_round.  With ``screen`` the
    shared node bases of csrc/nodepairs.cuh rule out the candidates that cannot win whenever E is dense in few nodes
    (the find_top_missing_edges case) and only the contenders take the exact path: the returned edge and value are
    those of the exact round either way.
    Returns (best, bestval, scores, exact_mask, info): best = row of E (-1: none); scores are exact where
    exact_mask is set and screen values (1e-9 .. 1e-8 relative) elsewhere; info = dict(exact, screened, nodes, levels)."""
    if miobi not in ("break", "make"):
        raise ValueError("KRYLOV_MIOBI:: not supported option for miobi")
    M = _mat(A)
    it = _default_it(M, it)
    E = np.asfortranarray(np.atleast_2d(np.asarray(E)).astype(np.int64))
    nE = E.shape[0]
    scores = np.zeros(nE)
    mask = np.zeros(nE, dtype=np.int32)
    info = np.zeros(4, dtype=np.int64)
    best, bestval = C.c_int64(), C.c_double()
    check(M.ctx.lib.kr_greedy_round(M.ctx.h, M.h, nE, _ptr(E), float(b_offdiag),
                                    float(b_offdiag if b_self is None else b_self), float(tol), it, fun_id(fun),
                                    0 if miobi == "break" else 1, int(bool(screen)), C.byref(best), C.byref(bestval),
                                    _ptr(scores), _ptr(mask), _ptr(info)))
    return (int(best.value), float(bestval.value), scores, mask.astype(bool),
            dict(exact=int(info[0]), screened=int(info[1]), nodes=int(info[2]), levels=int(info[3])))


def fun_update(A, U, B, fun, tol=1e-12, it=None, debug=0, nargout=3):
    """[Xm,iter,lucky,Um] = fun_update(A,U,B,fun,tol,it,debug)  (functions/fun_update.m:1-137).
    ``nargout`` = 4 selects the Arnoldi variant and returns the basis (fun_update.m:69,77)."""
    M = _mat(A)
    it = _default_it(M, it)
    if sp.issparse(U):
        U = U.toarray()
    U, ldu = _f64_cm(U)
    B, ldb = _f64_cm(np.atleast_2d(np.asarray(B, dtype=np.float64)))
    dim, k, lucky, dense = C.c_int64(), C.c_int64(), C.c_int(), C.c_int()
    lib = M.ctx.lib
    check(lib.kr_fun_update(M.ctx.h, M.h, U.shape[1], _ptr(U), ldu, _ptr(B), ldb, fun_id(fun), float(tol), it,
                            int(nargout >= 4), C.byref(dim), C.byref(k), C.byref(lucky), C.byref(dense)))
    d = dim.value
    Xm = np.empty((d, d), order="F")
    Um = np.empty((M.n, d), order="F") if nargout >= 4 else None
    check(lib.kr_fun_update_fetch(M.ctx.h, _ptr(Xm), max(d, 1), _ptr(Um), max(M.n, 1)))
    if not dense.value:
        if lucky.value:
            warnings.warn("FUN_UPDATE:: Detected lucky breakdown")
        if k.value == it:
            warnings.warn("FUN_UPDATE:: Reached maximum number of iterations")
    if nargout >= 4:
        return Xm, k.value, bool(lucky.value), Um
    return Xm, k.value, bool(lucky.value)


def function_multiple_entries(A, omega, f, tol=1e-12, it=None, poles=np.inf, debug=0):
    """[X,iter] = function_multiple_entries(A,omega,f,tol,it,poles,debug)
    (functions/function_multiple_entries.m:1-172)."""
    if not (np.isscalar(poles) and poles == np.inf):
        raise ValueError("FUNCTION_MULTIPLE_ENTRIES::Unsupported rational Krylov yet")
    M = _mat(A)
    it = _default_it(M, it)
    om = np.asfortranarray(np.atleast_2d(np.asarray(omega)).astype(np.int64))
    k = om.shape[0]
    X = np.zeros(k)
    itv = C.c_int64()
    check(M.ctx.lib.kr_function_multiple_entries(M.ctx.h, M.h, k, _ptr(om), fun_id(f), float(tol), it, _ptr(X),
                                                 C.byref(itv)))
    if itv.value == it:
        warnings.warn("FUNCTION_MULTIPLE_ENTRIES:: Reached maximum number of iterations")
    return X, itv.value


def trace_fun_sparse_update(A, X, Omega, fun, tol=1e-12, it=None, qmax=32, return_info=False):
    """(dtr, q, iter) with dtr = tr fun(A) - tr fun(A - D), D = Delta(X, Omega): D(i,j) = D(j,i) = X[h] for every row
    (i, j) of Omega (1-based; duplicates add up, a diagonal pair gives D(i,i) = X[h]) - so A here is the UPDATED matrix.
    kr_trace_fun_sparse_update: q-point Gauss-Legendre along A_t = A - (1 - t) D, each node one set of entries
    fun'(A_t)_Omega (function_multiple_entries' Krylov spaces with its tol and it); q is chosen from the quadrature's
    error bound against tol * sum_h c_h |X_h| and capped at min(qmax, 32); iter is the largest step count of any entry.
    Deterministic.  return_info adds {'tier_columns': [3 counts], 'dense_columns': count}, a column being one
    (start node, quadrature node) pair of the local path (csrc/entries_local.cuh)."""
    M = _mat(A)
    it = _default_it(M, it)
    Om = np.asfortranarray(np.asarray(Omega).reshape(-1, 2).astype(np.int64))
    X = np.ascontiguousarray(np.asarray(X, dtype=np.float64).ravel())
    if X.size != Om.shape[0]:
        raise ValueError("X must have one value per row of Omega")
    dtr = C.c_double()
    q = C.c_int64()
    itv = C.c_int64()
    info = (C.c_int64 * 4)()
    check(M.ctx.lib.kr_trace_fun_sparse_update(M.ctx.h, M.h, Om.shape[0], _ptr(Om), _ptr(X), fun_id(fun), float(tol),
                                               it, int(qmax), C.byref(dtr), C.byref(q), C.byref(itv), info))
    if return_info:
        return dtr.value, q.value, itv.value, {"tier_columns": list(info)[:3], "dense_columns": info[3]}
    return dtr.value, q.value, itv.value


def _fun_and_grad(X, A, Omega, fun, dfun, dfA, tol, it):
    M = _mat(A)
    X = np.ascontiguousarray(np.asarray(X, dtype=np.float64).ravel())
    Om = np.asfortranarray(np.atleast_2d(np.asarray(Omega)).astype(np.int64))
    dfA = np.ascontiguousarray(np.asarray(dfA, dtype=np.float64).ravel())
    f = C.c_double()
    gr = np.zeros(Om.shape[0])
    check(M.ctx.lib.kr_fun_and_grad_krylov(M.ctx.h, M.h, Om.shape[0], _ptr(X), _ptr(Om), fun_id(fun), fun_id(dfun),
                                           _ptr(dfA), float(tol), int(it), C.byref(f), _ptr(gr)))
    return f.value, gr


def fun_and_grad_krylov_exp(X, A, Omega, eA, tol, it, debug=False):
    """[f,gr] = fun_and_grad_krylov_exp(X,A,Omega,eA,tol,it,debug)
    (functions/fun_and_grad_krylov_exp.m:1-113)."""
    try:
        return _fun_and_grad(X, A, Omega, "exp", "exp", eA, tol, it)
    except Exception as e:
        if "not Hermitian" in str(e):
            raise ValueError("FUN_AND_GRAD_KRYLOV:: matrix A is not Hermitian")
        raise


def fun_and_grad_krylov_fun(X, A, Omega, fun, dfun, dfA, tol, it, debug=False, fun_M=None):
    """[f,gr] = fun_and_grad_krylov_fun(X,A,Omega,fun,dfun,dfA,tol,it,debug,fun_M)
    (functions/fun_and_grad_krylov_fun.m:1-71)."""
    if _is_exp(fun) and _is_exp(dfun):
        raise ValueError("use fun_and_grad_krylov_exp for f = exp (the reference's exp path shares one fun_update)")
    try:
        return _fun_and_grad(X, A, Omega, fun, dfun, dfA, tol, it)
    except Exception as e:
        if "not Hermitian" in str(e):
            raise ValueError("FUN_AND_GRAD_KRYLOV_FCONNECTIVITY:: matrix A is not Hermitian")
        raise


def normest(A, tol=1e-6):
    """MATLAB normest(A,tol) on the device SpMM (used at functions/fun_and_grad_krylov_fun.m:27)."""
    M = _mat(A)
    e, c = C.c_double(), C.c_int64()
    check(M.ctx.lib.kr_normest(M.ctx.h, M.h, float(tol), C.byref(e), C.byref(c)))
    return e.value, c.value


# ----------------------------------------------------------------------------- expmv family
def normAm(A, m):
    """[c,mv] = normAm(A,m)  (functions/normAm.m:1-52)."""
    M = _mat(A)
    c, mv = C.c_double(), C.c_int64()
    check(M.ctx.lib.kr_normAm(M.ctx.h, M.h, 1.0, int(m), C.byref(c), C.byref(mv)))
    return c.value, mv.value


def select_taylor_degree(A, b, m_max=55, p_max=8, prec="double", shift=False, bal=False, force_estm=False):
    """[M,mv,alpha,unA] = select_taylor_degree(A,b,m_max,p_max,prec,shift,bal,force_estm)
    (functions/select_taylor_degree.m:1-68).  Double precision, unbalanced only."""
    if prec != "double" or bal:
        raise NotImplementedError("device path: prec='double', bal=false only")
    m_max = 55 if m_max is None else int(m_max)
    p_max = 8 if p_max is None else int(p_max)
    if p_max < 2 or m_max > 60 or m_max + 1 < p_max * (p_max - 1):
        raise ValueError(">>> Invalid p_max or m_max.")
    M = _mat(A)
    ncols = 1 if np.ndim(b) == 1 else np.shape(b)[1]
    Mt = np.zeros((m_max, p_max - 1), order="F")
    alpha = np.zeros(p_max - 1)
    mv, unA = C.c_int64(), C.c_int()
    check(M.ctx.lib.kr_select_taylor_degree(M.ctx.h, M.h, 1.0, ncols, m_max, p_max, int(bool(shift)),
                                            int(bool(force_estm)), _ptr(Mt), C.byref(mv), _ptr(alpha), C.byref(unA)))
    return Mt, mv.value, alpha, unA.value


def expmv(t, A, b, M=None, prec="double", shift=True, bal=False, full_term=False, prnt=False):
    """[f,s,m,mv,mvd,unA] = expmv(t,A,b,M,prec,shift,bal,full_term,prnt)  (functions/expmv.m:1-94)."""
    if prec != "double" or bal:
        raise NotImplementedError("device path: prec='double', bal=false only")
    Mx = _mat(A)
    b, ldb = _f64_cm(b)
    if b.shape[0] != Mx.n:
        raise ValueError("The block vector b has wrong number of rows")
    f = np.empty_like(b, order="F")
    s, m, mv, mvd, unA = C.c_int64(), C.c_int64(), C.c_int64(), C.c_int64(), C.c_int()
    if M is not None:
        Mt, _ = _f64_cm(M)
        mm, pc = Mt.shape
    else:
        Mt, mm, pc = None, 0, 0
    check(Mx.ctx.lib.kr_expmv(Mx.ctx.h, Mx.h, float(t), b.shape[1], _ptr(b), ldb, _ptr(Mt), mm, pc, int(bool(shift)),
                              int(bool(full_term)), _ptr(f), ldb, C.byref(s), C.byref(m), C.byref(mv), C.byref(mvd),
                              C.byref(unA)))
    return f, s.value, m.value, mv.value, mvd.value, (None if M is not None else unA.value)


class ExpmvHandle:
    """Stands for the reference's handle ``@(x) expmv(1,A,x,[],'double')`` (functions/trace_exp.m:5)."""

    def __init__(self, A):
        self.M = _mat(A)

    def __call__(self, x):
        return expmv(1, self.M, x, None, "double")[0]


def mc_trace(Afun, n, tol=1e-3, maxit=10, isAreal=0, debug=0, probes=None):
    """[tr,res,it] = mc_trace(Afun,n,tol,maxit,isAreal,debug)  (functions/mc_trace.m:1-62), parity mode.
    Afun: a matrix (mc_trace.m:32-34) or an ExpmvHandle.  ``probes``: list of K = ceil(maxit/30) pairs
    (S, G) of n x 10 sign matrices - the reference draws them from an unseeded stream (:43-44)."""
    if isinstance(Afun, ExpmvHandle):
        M, op = Afun.M, 1
    elif isinstance(Afun, Matrix) or sp.issparse(Afun) or isinstance(Afun, np.ndarray):
        M, op = _mat(Afun), 0
    else:
        raise ValueError("mc_trace: the device path takes a matrix or an ExpmvHandle as Afun")
    K = int(math.ceil(maxit / 30))
    if probes is None or len(probes) < K:
        raise ValueError("mc_trace: pass K = ceil(maxit/30) = %d probe pairs (S, G)" % K)
    buf = np.empty((M.n, 20 * K), order="F")
    for i in range(K):
        buf[:, 20 * i:20 * i + 10] = probes[i][0]
        buf[:, 20 * i + 10:20 * i + 20] = probes[i][1]
    tr, res, it = C.c_double(), C.c_double(), C.c_int64()
    check(M.ctx.lib.kr_mc_trace(M.ctx.h, M.h, op, float(tol), int(maxit), _ptr(buf), C.byref(tr), C.byref(res),
                                C.byref(it)))
    return tr.value, res.value, it.value


def trace_exp(A, probes):
    """tr = trace_exp(A)  (functions/trace_exp.m:1-7); ``probes`` as in mc_trace (34 pairs)."""
    return mc_trace(ExpmvHandle(A), _mat(A).n, 1e-4, 1000, 1, probes=probes)[0]


# ----------------------------------------------------------------------------- greedy drivers (f1, f2)
def edge2low_rank(E, n, sign=-1.0):
    """[U,B] = edge2low_rank(E,n)  (functions/edge2low_rank.m:1-13); host-side glue."""
    E = np.atleast_2d(np.asarray(E)).astype(np.int64)
    ut = np.unique(E.ravel())
    pos = {int(a): i for i, a in enumerate(ut)}
    U = sp.csr_matrix((np.ones(ut.size), (ut - 1, np.arange(ut.size))), shape=(n, ut.size))
    B = np.zeros((ut.size, ut.size))
    for a, b in E:
        B[pos[int(a)], pos[int(b)]] = sign
        B[pos[int(b)], pos[int(a)]] = sign
    return U, B


def compute_centrality(A, kind="eig", tol=1e-13, maxit=20000):
    """c = compute_centrality(A,type)  (functions/compute_centrality.m:1-32).

    'eig' (:15-17, the reference calls eigs(A,1)) and 'pr' (:20-26, PageRank with alpha = 0.85) are power
    iterations that run entirely on the device (kr_compute_centrality: one kernel launch for the reference's
    graph sizes, stopping test included); 'deg' (:18-19) is a column sum; 'exp' (:9-10, diag(expm(A))) goes
    through function_multiple_entries on the diagonal pairs.  'res' (:11-14) uses an undefined `n` in the
    reference and raises there too.  Unknown types fall back to 'eig' with the reference's notice (:27-30)."""
    if kind == "deg":
        return np.asarray(sp.csr_matrix(A).sum(axis=0)).ravel()
    if kind == "res":
        raise NameError("compute_centrality: 'res' references an undefined variable n in the reference "
                        "(functions/compute_centrality.m:14)")
    M = _mat(A)
    if kind == "exp":
        idx = np.arange(1, M.n + 1, dtype=np.int64)
        nrm = normest(M, 1e-2)[0]
        return function_multiple_entries(M, np.stack([idx, idx], axis=1), "exp", 1e-13 * math.exp(nrm), None)[0]
    if kind not in ("eig", "pr"):
        print("#### Centrality set to eig ####")
        kind = "eig"
    c = np.zeros(M.n)
    iters, conv = C.c_int64(), C.c_int()
    check(M.ctx.lib.kr_compute_centrality(M.ctx.h, M.h, 0 if kind == "eig" else 1, float(tol), int(maxit), _ptr(c),
                                          C.byref(iters), C.byref(conv)))
    return c


def _tril_edges(A):
    L = sp.tril(sp.csc_matrix(A), k=-1, format="csc")
    L.sort_indices()
    L.eliminate_zeros()
    J = np.repeat(np.arange(L.shape[1]), np.diff(L.indptr)) + 1
    return (L.indices + 1).astype(np.int64), J.astype(np.int64)


def find_top_edges(A, centrality, num, order="mult"):
    """E = find_top_edges(A,centrality,num,order)  (functions/find_top_edges.m:1-40); index bookkeeping."""
    centrality = np.asarray(centrality, dtype=np.float64).ravel()
    I, J = _tril_edges(A)
    E = np.stack([I, J], axis=1)
    if I.size < num:
        warnings.warn("FIND_TOP_EDGES:: there are not enough edges in the graph")
    if order == "mult":
        ind = np.argsort(-(centrality[I - 1] * centrality[J - 1]), kind="stable")
        return E[ind[:num]]
    if order == "min":
        sc = np.sort(centrality)
        rank = lambda v: sc.size - np.searchsorted(sc, v, side="right") + 1
        c1, c2 = rank(centrality[I - 1]), rank(centrality[J - 1])
        mn = np.minimum(c1, c2).astype(np.float64)
        mx = np.maximum(c1, c2).astype(np.float64)
        ind = np.argsort(mx * (mx - 1) / 2 + mn, kind="stable")
        return E[ind[:num]]
    raise ValueError(order)


def find_top_missing_edges(A, centrality, num, order="min"):
    """E = find_top_missing_edges(A,centrality,num,order)  (functions/find_top_missing_edges.m:1-67):
    'min' (:55-65, the ordering the reference's scripts use) and 'mult' (:20-54)."""
    centrality = np.asarray(centrality, dtype=np.float64).ravel()
    indC = np.argsort(-centrality, kind="stable")
    Ac = sp.csc_matrix(A)
    n = Ac.shape[0]

    def missing_above(j):
        """nodes ranked before the j-th (1-based) that are NOT adjacent to it, in rank order"""
        col = np.zeros(n)
        s, e = Ac.indptr[indC[j - 1]], Ac.indptr[indC[j - 1] + 1]
        col[Ac.indices[s:e]] = Ac.data[s:e]
        cand = indC[:j - 1]
        return cand[col[cand] == 0]

    if order == "min":
        rows, total, j = [], 0, 2
        while total < num:
            ind = missing_above(j)
            rows.append(np.stack([ind + 1, np.full(ind.size, indC[j - 1] + 1)], axis=1))
            total += ind.size
            j += 1
        return np.concatenate(rows, axis=0)[:num].astype(np.int64)
    if order != "mult":
        raise ValueError("find_top_missing_edges: order must be 'mult' or 'min'")
    if (n * n - Ac.nnz - n) / 2 <= num:
        # :21-29 returns without assigning E in the reference (an error there as well)
        raise ValueError("find_top_missing_edges: not enough missing edges for order 'mult'")
    sc = centrality[indC]
    # smallest prefix of the ranking that already contains `num` missing edges (:31-37)
    prefix, found = 2, 0
    while found < num:
        found += missing_above(prefix).size
        prefix += 1
    prefix -= 1
    # every pair whose product can beat the weakest pair of that prefix lies among the first N nodes (:39)
    N = int(np.count_nonzero(sc[0] * sc > sc[prefix - 1] ** 2))
    S = np.triu(np.outer(sc[:N], sc[:N]))
    flat = np.argsort(-S.ravel(order="F"), kind="stable")               # sort(S(:), 'descend'): column-major, stable
    ii, jj = np.unravel_index(flat, S.shape, order="F")
    sub = Ac[indC[:N], :][:, indC[:N]].toarray()
    keep = (ii != jj) & (sub[ii, jj] == 0)
    ii, jj = ii[keep][:num], jj[keep][:num]
    return np.stack([indC[ii] + 1, indC[jj] + 1], axis=1).astype(np.int64)


def _issymmetric(A):
    A = sp.csr_matrix(A)
    return (A != A.T).nnz == 0


def select_candidate(vals, miobi):
    """First-wins strict comparison of functions/krylov_miobi.m:112-124."""
    vals = np.asarray(vals, dtype=np.float64)
    # a strict comparison against +-inf skips NaN and infinities of the wrong sign; argmin / argmax return the FIRST
    # extremum, i.e. the reference's first-wins rule
    key = np.where(np.isnan(vals), np.inf, vals) if miobi == "break" else np.where(np.isnan(vals), -np.inf, vals)
    if key.size == 0:
        return -1, (np.inf if miobi == "break" else -np.inf)
    best = int(np.argmin(key)) if miobi == "break" else int(np.argmax(key))
    if not (key[best] < np.inf if miobi == "break" else key[best] > -np.inf):
        return -1, (np.inf if miobi == "break" else -np.inf)
    return best, float(vals[best])


def krylov_miobi(A, k, E=None, tol=1e-12, it=None, poles=np.inf, debug=0, miobi="break", rescale=1.0, scorer=None,
                 screen=False):
    """[edges,rob,A_new] = krylov_miobi(A,k,E,tol,it,poles,debug,miobi,rescale)
    (functions/krylov_miobi.m:1-142).  The candidate loop (:76-99) is one batched device call;
    ``scorer(M, E, b_offdiag, tol, it)`` may replace it (multi-GPU sharding, tests); ``screen`` runs each round
    through greedy_round (candidates that cannot win are ruled out by shared node bases, the winner is exact)."""
    if not _issymmetric(A):
        raise ValueError("KRYLOV_MIOBI:: Adjacency matrix should be symmetric")
    if miobi not in ("break", "make"):
        raise ValueError("KRYLOV_MIOBI:: not supported option for miobi")
    A = sp.csr_matrix(A).astype(np.float64)
    if miobi == "break" and A.nnz < 2 * k:
        raise ValueError("KRYLOV_MIOBI:: edges to be removed are more than edges in the network")
    n = A.shape[0]
    it = int(min(100, n)) if it is None else int(it)
    if E is None or len(E) == 0:
        Ac = sp.coo_matrix(A)
        keep = Ac.row >= Ac.col
        order = np.lexsort((Ac.row[keep], Ac.col[keep]))
        E = np.stack([Ac.row[keep][order] + 1, Ac.col[keep][order] + 1], axis=1)
    E = np.atleast_2d(np.asarray(E)).astype(np.int64)
    sign = -1.0 if miobi == "break" else 1.0
    M = Matrix(A)
    rob, edges = 0.0, np.zeros((0, 2), dtype=np.int64)
    for _ in range(min(k, E.shape[0])):
        if scorer is not None:
            vals = np.asarray(scorer(M, E, sign / rescale, tol, it))
            best, bestval = select_candidate(vals, miobi)
        elif screen:
            best, bestval = greedy_round(M, E, sign / rescale, tol, it, "exp", miobi, True, b_self=sign)[:2]
        else:
            vals = trace_fun_update_edges(M, E, sign / rescale, tol, it, "exp", b_self=sign)[0]
            best, bestval = select_candidate(vals, miobi)
        chosen = E[best].copy()
        E = np.delete(E, best, axis=0)
        newval = 0.0 if miobi == "break" else 1.0
        M.set_edges([chosen[0]], [chosen[1]], newval)                    # :129-135 on the device copy
        A = A.tolil()
        A[chosen[0] - 1, chosen[1] - 1] = newval
        A[chosen[1] - 1, chosen[0] - 1] = newval
        A = A.tocsr()
        A.eliminate_zeros()
        edges = np.vstack([edges, chosen[None, :]])
        rob += bestval
    return edges, rob, A


def greedy_krylov(A, k, Q=0, centrality=None, order="mult", tol=1e-12, it=None, poles=np.inf, debug=0, miobi="break",
                  rescale=1.0, scorer=None, screen=False):
    """[edges,rob_variation,A_new] = greedy_krylov(A,k,Q,centrality,order,tol,it,poles,debug,miobi,rescale)
    (functions/greedy_krylov.m:1-97).  A stays resident on the device across the k rounds; each round is
    one batched scoring call plus an in-place edge update."""
    if not _issymmetric(A):
        raise ValueError("GREEDY_KRYLOV:: Adjacency matrix should be symmetric")
    A = sp.csr_matrix(A).astype(np.float64)
    n = A.shape[0]
    it = int(min(100, n)) if it is None else int(it)
    if not Q:
        Q = int(np.asarray(A.sum(axis=0)).max())
    if miobi == "break" and A.nnz < 2 * k:
        raise ValueError("GREEDY_KRYLOV:: edges to be removed are more than edges in the network")
    sign = -1.0 if miobi == "break" else 1.0
    newval = 0.0 if miobi == "break" else 1.0
    M = Matrix(A)
    A = A.tolil()
    rob_variation, edges = 0.0, np.zeros((0, 2), dtype=np.int64)
    top_edges, chosen = None, None
    for j in range(1, k + 1):
        if j == 1:
            top_edges = (find_top_missing_edges if miobi == "make" else find_top_edges)(A.tocsr(), centrality, Q + k,
                                                                                        order)
        else:
            top_edges = top_edges[~np.all(top_edges == chosen, axis=1)]      # :84-86
        E = top_edges[:Q]
        if scorer is not None:
            vals = np.asarray(scorer(M, E, sign / rescale, tol, it))
            best, bestval = select_candidate(vals, miobi)
        elif screen:
            best, bestval = greedy_round(M, E, sign / rescale, tol, it, "exp", miobi, True, b_self=sign)[:2]
        else:
            vals = trace_fun_update_edges(M, E, sign / rescale, tol, it, "exp", b_self=sign)[0]
            best, bestval = select_candidate(vals, miobi)
        chosen = E[best].copy()
        M.set_edges([chosen[0]], [chosen[1]], newval)
        A[chosen[0] - 1, chosen[1] - 1] = newval
        A[chosen[1] - 1, chosen[0] - 1] = newval
        edges = np.vstack([edges, chosen[None, :]])
        rob_variation += bestval
    A = A.tocsr()
    A.eliminate_zeros()
    return edges, rob_variation, A


def greedy_krylov_nodes(A, k, Q=0, centrality=None, tol=1e-12, it=None, fun="exp"):
    """[nodes,rob_variation,A_new]: greedy node attack, the node counterpart of greedy_krylov (functions/greedy_krylov.m).
    Round 1 ranks the nodes by centrality (descending, stable) and keeps the top Q + k; every round scores the first Q
    remaining nodes in one trace_fun_update_nodes call, takes the first-wins arg-min (select_candidate(..., 'break')),
    deletes the chosen node's off-diagonal entries with one in-place set_edges call and drops it from the list.  A stays
    on the device across the rounds.  Q = 0 takes the reference's default, the largest column sum of A; centrality =
    None computes the 'eig' centrality on the device.  Returns nodes (1-based), the summed scores and the edited A."""
    if not _issymmetric(A):
        raise ValueError("GREEDY_KRYLOV:: Adjacency matrix should be symmetric")
    A = sp.csr_matrix(A).astype(np.float64)
    n = A.shape[0]
    it = int(min(100, n)) if it is None else int(it)
    if not Q:
        Q = int(np.asarray(A.sum(axis=0)).max())
    M = Matrix(A)
    if centrality is None:
        centrality = compute_centrality(M, "eig")
    top = np.argsort(-np.asarray(centrality, dtype=np.float64).ravel(), kind="stable")[:Q + k] + 1
    A = A.tolil()
    nodes, rob_variation = [], 0.0
    for _ in range(min(k, top.size)):
        cand = top[:Q]
        vals = trace_fun_update_nodes(M, cand, tol, it, fun)[0]
        best, bestval = select_candidate(vals, "break")
        chosen = int(cand[best])
        nbrs = [j + 1 for j in A.rows[chosen - 1] if j != chosen - 1]
        if nbrs:
            M.set_edges(np.full(len(nbrs), chosen), nbrs, 0.0)
            for j in nbrs:
                A[chosen - 1, j - 1] = 0.0
                A[j - 1, chosen - 1] = 0.0
        top = top[top != chosen]
        nodes.append(chosen)
        rob_variation += bestval
    A = A.tocsr()
    A.eliminate_zeros()
    return np.asarray(nodes, dtype=np.int64), rob_variation, A


def fun_and_grad_all_edges(X, A, Omega, fun, dfun, tol=1e-8, it=None, objective=False):
    """Objective and gradient over a LARGE edge set Omega (config C2: "gradient over all edges").

    Calling fun_and_grad_krylov_fun literally with Omega = all edges makes U an n x n selector and the
    reference falls into its dense branch (functions/fun_update.m:85-90; SURVEY.md note N1).  The
    mathematically identical sparse formulation used by the reference's own Hessian callback
    (functions/hessianfcn_fun.m:5-7) is evaluated instead:
        Atilde = A + Delta(X, Omega),   gr = -2 * dfun(Atilde)_Omega   (function_multiple_entries, one
        single-vector Krylov space per distinct row, all advanced by one wide SpMM per step).
    With objective=True the objective f = -(trace fun(Atilde) - trace fun(A)) comes too, from
    trace_fun_sparse_update on the same device copy of Atilde with the same tol and it: a quadrature of the entries
    fun'(A_t)_Omega along the path from A to Atilde (deterministic, to tol; the derivative is taken from fun, dfun
    serves the gradient only).  Returns gr (len(Omega)), or (f, gr) with objective=True."""
    A = sp.csr_matrix(A).astype(np.float64)
    n = A.shape[0]
    Om = np.atleast_2d(np.asarray(Omega)).astype(np.int64)
    X = np.asarray(X, dtype=np.float64).ravel()
    D = sp.csr_matrix((X, (Om[:, 0] - 1, Om[:, 1] - 1)), shape=(n, n))
    At = (A + D + D.T).tocsr()
    if not objective:
        vals, _ = function_multiple_entries(At, Om, dfun, tol, it)
        return -2.0 * vals
    Mt = Matrix(At)
    vals, _ = function_multiple_entries(Mt, Om, dfun, tol, it)
    # D + D' above puts 2 X_h on the diagonal for a pair (i, i); Delta of trace_fun_sparse_update puts X_h there
    Xd = np.where(Om[:, 0] == Om[:, 1], 2.0 * X, X)
    dtr = trace_fun_sparse_update(Mt, Xd, Om, fun, tol, it)[0]
    return -dtr, -2.0 * vals


def _hessian(X, A, Omega, fun, tol, it):
    A = sp.csr_matrix(A).astype(np.float64)
    n = A.shape[0]
    Om = np.asfortranarray(np.atleast_2d(np.asarray(Omega)).astype(np.int64))
    X = np.asarray(X, dtype=np.float64).ravel()
    XX = sp.csr_matrix((X, (Om[:, 0] - 1, Om[:, 1] - 1)), shape=(n, n))
    M = Matrix((A + XX + XX.T).tocsr())                   # Atilde (functions/hessianfcn_exp.m:4-7)
    m = Om.shape[0]
    Hes = np.zeros((m, m), order="F")
    itv = C.c_int64()
    check(M.ctx.lib.kr_frechet_hessian(M.ctx.h, M.h, m, _ptr(Om), fun_id(fun), float(tol), int(it), _ptr(Hes),
                                       C.byref(itv)))
    if itv.value == int(it):
        warnings.warn("MULTIPLE_FRECHET_EVAL:: Reached maximum number of iterations")
    return Hes


def hessp_all_edges(X, A, Omega, f, Y, tol=1e-8, it=None, reference_form=False, return_info=False):
    """W = Hes * Y for the all-edges callbacks without assembling Hes (fmincon's HessianMultiplyFcn, SciPy's hessp):
    kr_frechet_hessian_multiply on Atilde = A + Delta(X, Omega) (assembled as in hessianfcn_fun.m:4-7), or on A itself
    when A is a resident Matrix of Atilde (X is then not used).  f is the function whose Frechet derivative is taken,
    dfun of the gradient.  The default is the Hessian of the objective -(tr fun(Atilde) - tr fun(A)), whose gradient
    fun_and_grad_all_edges returns; reference_form=True gives hessianfcn_fun's matrix times Y, which leaves out the
    term of the mirrored direction e_b e_a' (DESIGN.md section 2).  Y is 1-D (returns 1-D) or len(Omega) x p.
    return_info adds (iter, {'tier_pairs': [3 counts], 'dense_pairs': count})."""
    Om = np.asfortranarray(np.asarray(Omega).reshape(-1, 2).astype(np.int64))
    m = Om.shape[0]
    if isinstance(A, Matrix):
        M = A
    else:
        A = sp.csr_matrix(A).astype(np.float64)
        n = A.shape[0]
        X = np.asarray(X, dtype=np.float64).ravel()
        XX = sp.csr_matrix((X, (Om[:, 0] - 1, Om[:, 1] - 1)), shape=(n, n))
        M = Matrix((A + XX + XX.T).tocsr())
    it = _default_it(M, it)
    Y = np.asarray(Y, dtype=np.float64)
    vec = Y.ndim == 1
    if Y.ndim not in (1, 2) or Y.shape[0] != m:
        raise ValueError("Y must have one row per row of Omega")
    Yc = np.asfortranarray(Y.reshape(m, -1))
    p = Yc.shape[1]
    W = np.zeros((m, p), order="F")
    itv = C.c_int64()
    info = (C.c_int64 * 4)()
    check(M.ctx.lib.kr_frechet_hessian_multiply(M.ctx.h, M.h, m, _ptr(Om), p, _ptr(Yc), max(m, 1), fun_id(f),
                                                1 if reference_form else 0, float(tol), it, _ptr(W), max(m, 1),
                                                C.byref(itv), info))
    if itv.value == min(it, 64):
        warnings.warn("MULTIPLE_FRECHET_EVAL:: Reached maximum number of iterations")
    W = W[:, 0] if vec else W
    if return_info:
        return W, itv.value, {"tier_pairs": list(info)[:3], "dense_pairs": info[3]}
    return W


def hessianfcn_exp(X, A, Omega, tol, it):
    """Hes = hessianfcn_exp(X,A,Omega,tol,it)  (functions/hessianfcn_exp.m:1-17)."""
    return _hessian(X, A, Omega, "exp", tol, it)


def hessianfcn_fun(X, A, Omega, f, tol, it):
    """Hes = hessianfcn_fun(X,A,Omega,f,tol,it)  (functions/hessianfcn_fun.m:1-17)."""
    return _hessian(X, A, Omega, f, tol, it)
