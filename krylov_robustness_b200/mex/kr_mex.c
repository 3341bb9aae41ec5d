/*
 * kr_mex.c - single MEX gateway (string-dispatched) from MATLAB / GNU Octave into the C ABI of
 * libkrylov_b200.so (include/krylov_b200.h).  The wrappers in ../matlab/ keep the reference's
 * function signatures and call   varargout = kr_mex('<op>', args...).
 *
 * The build image has neither mex.h nor mkoctfile (SURVEY.md section 0); tests/test_mex_gateway.py
 * compiles this file against a stub of the MEX API (tests/mex_stub/) and runs it on the GPU tier.  It is
 * a thin marshaller on purpose - every line with arithmetic in it lives behind the C ABI and is
 * exercised from Python (tests/).  Build where MATLAB/Octave exists:
 *   mex -I../../include kr_mex.c -L.. -lkrylov_b200          (MATLAB)
 *   mkoctfile --mex -I../../include kr_mex.c -L.. -lkrylov_b200   (Octave)
 *
 * Sparse A arrives as MATLAB CSC (Jc, Ir, Pr).  Every A on this path is symmetric
 * (functions/greedy_krylov.m:27, functions/krylov_miobi.m:26, functions/fun_and_grad_krylov_fun.m:22),
 * so its CSC arrays are its CSR arrays and are passed through unchanged; an unsymmetric A is
 * transposed by the wrapper (A.') before the call.  Device copies of A are cached, keyed on (n, nnz, a 64-bit
 * fingerprint of the CONTENT of Jc / Ir / Pr): MATLAB re-uses freed addresses, so the data pointer identifies
 * nothing (a fresh `A + XX + XX'` of the Hessian callbacks lands on the old address with the same pattern and
 * nnz).  Krylov state handles are tracked here too; both are released by mexAtExit.
 */
#include <string.h>
#include <stdlib.h>
#include "mex.h"
#include "krylov_b200.h"

static kr_ctx* g_ctx = NULL;
#define KR_CACHE 8
static struct { uint64_t key; mwSize n, nnz; kr_matrix* M; } g_cache[KR_CACHE];
static int g_next = 0;
#define KR_MAX_KRYLOV 4096
static kr_krylov* g_krylov[KR_MAX_KRYLOV];      /* live Krylov handles (freed by 'krylov_free' or at exit) */
#define KR_MAX_MATS 64
static kr_matrix* g_mats[KR_MAX_MATS];          /* explicit matrix handles ('matrix_create' / 'matrix_free') */

static void at_exit(void) {
    int i;
    for (i = 0; i < KR_MAX_KRYLOV; ++i) if (g_krylov[i]) { kr_krylov_destroy(g_krylov[i]); g_krylov[i] = NULL; }
    for (i = 0; i < KR_CACHE; ++i) if (g_cache[i].M) { kr_matrix_destroy(g_cache[i].M); g_cache[i].M = NULL; }
    for (i = 0; i < KR_MAX_MATS; ++i) if (g_mats[i]) { kr_matrix_destroy(g_mats[i]); g_mats[i] = NULL; }
    if (g_ctx) { kr_ctx_destroy(g_ctx); g_ctx = NULL; }
}

static void track_krylov(kr_krylov* st) {
    int i;
    for (i = 0; i < KR_MAX_KRYLOV; ++i) if (!g_krylov[i]) { g_krylov[i] = st; return; }
    kr_krylov_destroy(st);
    mexErrMsgTxt("krylov_b200: too many live Krylov handles (clear the params structs that are no longer needed)");
}
static int untrack_krylov(kr_krylov* st) {      /* 1 if the handle was live */
    int i;
    for (i = 0; i < KR_MAX_KRYLOV; ++i) if (g_krylov[i] == st) { g_krylov[i] = NULL; return 1; }
    return 0;
}
static kr_krylov* live_krylov(const mxArray* h) {
    kr_krylov* st = *(kr_krylov**)mxGetData(h);
    int i;
    for (i = 0; i < KR_MAX_KRYLOV; ++i) if (st && g_krylov[i] == st) return st;
    mexErrMsgTxt("krylov_b200: stale or foreign Krylov handle");
    return NULL;
}

/* 64-bit content fingerprint (four interleaved multiply-xor lanes over 8-byte words) */
static uint64_t mix64(uint64_t h, uint64_t x) {
    h ^= x;
    h *= 0x9E3779B97F4A7C15ull;
    return h ^ (h >> 29);
}
static uint64_t hash_words(uint64_t seed, const void* data, size_t bytes) {
    const uint64_t* w = (const uint64_t*)data;
    size_t k = bytes / 8, i = 0;
    uint64_t h0 = seed, h1 = seed ^ 0xA0761D6478BD642Full, h2 = seed ^ 0xE7037ED1A0B428DBull, h3 = seed ^ 0x8EBC6AF09C88C6E3ull;
    for (; i + 4 <= k; i += 4) { h0 = mix64(h0, w[i]); h1 = mix64(h1, w[i + 1]); h2 = mix64(h2, w[i + 2]); h3 = mix64(h3, w[i + 3]); }
    for (; i < k; ++i) h0 = mix64(h0, w[i]);
    return mix64(mix64(mix64(h0, h1), h2), h3);
}

static void chk(int status) {
    if (status != 0) mexErrMsgIdAndTxt("krylov_b200:error", "%s", kr_last_error());
}

static kr_ctx* ctx(void) {
    if (!g_ctx) { chk(kr_ctx_create(0, &g_ctx)); mexAtExit(at_exit); }
    return g_ctx;
}

static kr_matrix* create_matrix(const mxArray* A);

/* The matrix argument of every op: a sparse A (device copy cached by content) or a uint64 handle from
 * 'matrix_create' (a device-resident matrix that 'matrix_set_edges' edits in place, functions/krylov_miobi.m:127-135). */
static kr_matrix* matrix_of(const mxArray* A) {
    int i;
    mwSize n, nnz;
    const mwIndex *jc, *ir;
    kr_matrix* M = NULL;
    uint64_t key;
    if (mxIsUint64(A)) {
        M = *(kr_matrix**)mxGetData(A);
        for (i = 0; i < KR_MAX_MATS; ++i) if (M && g_mats[i] == M) return M;
        mexErrMsgTxt("krylov_b200: stale or foreign matrix handle");
    }
    if (!mxIsSparse(A) || !mxIsDouble(A)) mexErrMsgTxt("A must be a real sparse double matrix");
    if (mxGetM(A) != mxGetN(A)) mexErrMsgTxt("The matrix A should be square");
    n = mxGetN(A); jc = mxGetJc(A); ir = mxGetIr(A); nnz = jc[n];
    key = hash_words(0x243F6A8885A308D3ull ^ (uint64_t)n, jc, (n + 1) * sizeof(mwIndex));
    key = hash_words(key, ir, nnz * sizeof(mwIndex));
    key = hash_words(key, mxGetPr(A), nnz * sizeof(double));
    for (i = 0; i < KR_CACHE; ++i)
        if (g_cache[i].M && g_cache[i].key == key && g_cache[i].n == n && g_cache[i].nnz == nnz) return g_cache[i].M;
    M = create_matrix(A);
    if (g_cache[g_next].M) kr_matrix_destroy(g_cache[g_next].M);
    g_cache[g_next].key = key; g_cache[g_next].n = n; g_cache[g_next].nnz = nnz; g_cache[g_next].M = M;
    g_next = (g_next + 1) % KR_CACHE;
    return M;
}

static kr_matrix* create_matrix(const mxArray* A) {
    mwSize n, nnz, p;
    const mwIndex *jc, *ir;
    int64_t *rp, *ci;
    kr_matrix* M = NULL;
    if (!mxIsSparse(A) || !mxIsDouble(A)) mexErrMsgTxt("A must be a real sparse double matrix");
    if (mxGetM(A) != mxGetN(A)) mexErrMsgTxt("The matrix A should be square");
    n = mxGetN(A); jc = mxGetJc(A); ir = mxGetIr(A); nnz = jc[n];
    rp = (int64_t*)mxMalloc((n + 1) * sizeof(int64_t));
    ci = (int64_t*)mxMalloc((nnz ? nnz : 1) * sizeof(int64_t));
    for (p = 0; p <= n; ++p) rp[p] = (int64_t)jc[p];
    for (p = 0; p < nnz; ++p) ci[p] = (int64_t)ir[p];
    chk(kr_matrix_create(ctx(), (int64_t)n, (int64_t)nnz, rp, ci, mxGetPr(A), &M));
    mxFree(rp); mxFree(ci);
    return M;
}

static int fun_of(const mxArray* f) {          /* wrapper passes func2str(f) */
    char buf[32];
    mxGetString(f, buf, sizeof buf);
    if (!strcmp(buf, "exp")) return KR_FUN_EXP;
    if (!strcmp(buf, "sinh")) return KR_FUN_SINH;
    if (!strcmp(buf, "cosh")) return KR_FUN_COSH;
    mexErrMsgTxt("krylov_b200: supported function handles are @exp, @sinh, @cosh");
    return -1;
}

static int64_t* to_i64(const mxArray* a, mwSize* count) {
    mwSize i, k = mxGetNumberOfElements(a);
    const double* p = mxGetPr(a);
    int64_t* out = (int64_t*)mxMalloc((k ? k : 1) * sizeof(int64_t));
    for (i = 0; i < k; ++i) out[i] = (int64_t)p[i];
    if (count) *count = k;
    return out;
}

static mxArray* scalar(double v) { return mxCreateDoubleScalar(v); }

void mexFunction(int nlhs, mxArray* plhs[], int nrhs, const mxArray* prhs[]) {
    char op[64];
    if (nrhs < 1 || mxGetString(prhs[0], op, sizeof op)) mexErrMsgTxt("kr_mex('<op>', ...)");
    prhs++; nrhs--;

    if (!strcmp(op, "matrix_create")) {                            /* h = kr_mex('matrix_create', A) */
        int i;
        kr_matrix* M = create_matrix(prhs[0]);
        for (i = 0; i < KR_MAX_MATS && g_mats[i]; ++i) {}
        if (i == KR_MAX_MATS) { kr_matrix_destroy(M); mexErrMsgTxt("krylov_b200: too many live matrix handles"); }
        g_mats[i] = M;
        plhs[0] = mxCreateNumericMatrix(1, 1, mxUINT64_CLASS, mxREAL);
        *(kr_matrix**)mxGetData(plhs[0]) = M;
    } else if (!strcmp(op, "matrix_free")) {                       /* kr_mex('matrix_free', h)  (idempotent) */
        int i;
        kr_matrix* M = *(kr_matrix**)mxGetData(prhs[0]);
        for (i = 0; i < KR_MAX_MATS; ++i) if (M && g_mats[i] == M) { kr_matrix_destroy(M); g_mats[i] = NULL; }
    } else if (!strcmp(op, "matrix_set_edges")) {                  /* kr_mex('matrix_set_edges', h, i, j, v): A(i,j) = A(j,i) = v */
        kr_matrix* M = matrix_of(prhs[0]);
        mwSize cnt = 0, cj = 0, q;
        int64_t* ii = to_i64(prhs[1], &cnt);
        int64_t* jj = to_i64(prhs[2], &cj);
        double* v = (double*)mxMalloc((cnt ? cnt : 1) * sizeof(double));
        if (cj != cnt) mexErrMsgTxt("matrix_set_edges: i and j must have the same length");
        for (q = 0; q < cnt; ++q) v[q] = mxGetNumberOfElements(prhs[3]) == 1 ? mxGetScalar(prhs[3]) : mxGetPr(prhs[3])[q];
        if (!mxIsUint64(prhs[0])) mexErrMsgTxt("matrix_set_edges needs a handle from matrix_create (a cached copy of a MATLAB matrix must not diverge from it)");
        chk(kr_matrix_set_edges(M, (int64_t)cnt, ii, jj, v));
        mxFree(ii); mxFree(jj); mxFree(v);
    } else if (!strcmp(op, "spmm")) {                              /* Y = kr_mex('spmm', A, X) */
        kr_matrix* M = matrix_of(prhs[0]);
        mwSize n = mxGetM(prhs[1]), k = mxGetN(prhs[1]);
        plhs[0] = mxCreateDoubleMatrix(n, k, mxREAL);
        chk(kr_spmm(ctx(), M, (int64_t)k, mxGetPr(prhs[1]), (int64_t)n, mxGetPr(plhs[0]), (int64_t)n));
    } else if (!strcmp(op, "trace_fun_update")) {                  /* [Xm,iter,lucky] = (A,U,B,tol,it,fun) */
        kr_matrix* M = matrix_of(prhs[0]);
        double x; int64_t it; int lucky;
        chk(kr_trace_fun_update(ctx(), M, (int64_t)mxGetN(prhs[1]), mxGetPr(prhs[1]), (int64_t)mxGetM(prhs[1]),
                                mxGetPr(prhs[2]), (int64_t)mxGetM(prhs[2]), mxGetScalar(prhs[3]),
                                (int64_t)mxGetScalar(prhs[4]), fun_of(prhs[5]), &x, &it, &lucky));
        plhs[0] = scalar(x);
        if (nlhs > 1) plhs[1] = scalar((double)it);
        if (nlhs > 2) plhs[2] = mxCreateLogicalScalar(lucky != 0);
    } else if (!strcmp(op, "trace_fun_update_edges")) {            /* [Xm,iter,lucky] = (A,E,b,tol,it,fun[,b_self]) */
        kr_matrix* M = matrix_of(prhs[0]);
        mwSize nE = mxGetM(prhs[1]), i;
        int64_t* E = to_i64(prhs[1], NULL);
        int64_t* it = (int64_t*)mxMalloc((nE ? nE : 1) * sizeof(int64_t));
        int* lk = (int*)mxMalloc((nE ? nE : 1) * sizeof(int));
        plhs[0] = mxCreateDoubleMatrix(nE, 1, mxREAL);
        chk(kr_trace_fun_update_edges_ex(ctx(), M, (int64_t)nE, E, mxGetScalar(prhs[2]),
                                         nrhs > 6 ? mxGetScalar(prhs[6]) : mxGetScalar(prhs[2]), mxGetScalar(prhs[3]),
                                         (int64_t)mxGetScalar(prhs[4]), fun_of(prhs[5]), mxGetPr(plhs[0]), it, lk));
        if (nlhs > 1) { plhs[1] = mxCreateDoubleMatrix(nE, 1, mxREAL); for (i = 0; i < nE; ++i) mxGetPr(plhs[1])[i] = (double)it[i]; }
        if (nlhs > 2) { plhs[2] = mxCreateDoubleMatrix(nE, 1, mxREAL); for (i = 0; i < nE; ++i) mxGetPr(plhs[2])[i] = (double)lk[i]; }
        mxFree(E); mxFree(it); mxFree(lk);
    } else if (!strcmp(op, "trace_fun_update_nodes")) {            /* [Xm,iter,lucky] = (A,V,tol,it,fun): node removal */
        kr_matrix* M = matrix_of(prhs[0]);
        mwSize nV = 0, i;
        int64_t* V = to_i64(prhs[1], &nV);
        int64_t* it = (int64_t*)mxMalloc((nV ? nV : 1) * sizeof(int64_t));
        int* lk = (int*)mxMalloc((nV ? nV : 1) * sizeof(int));
        plhs[0] = mxCreateDoubleMatrix(nV, 1, mxREAL);
        chk(kr_trace_fun_update_nodes(ctx(), M, (int64_t)nV, V, mxGetScalar(prhs[2]), (int64_t)mxGetScalar(prhs[3]),
                                      fun_of(prhs[4]), mxGetPr(plhs[0]), it, lk));
        if (nlhs > 1) { plhs[1] = mxCreateDoubleMatrix(nV, 1, mxREAL); for (i = 0; i < nV; ++i) mxGetPr(plhs[1])[i] = (double)it[i]; }
        if (nlhs > 2) { plhs[2] = mxCreateDoubleMatrix(nV, 1, mxREAL); for (i = 0; i < nV; ++i) mxGetPr(plhs[2])[i] = (double)lk[i]; }
        mxFree(V); mxFree(it); mxFree(lk);
    } else if (!strcmp(op, "greedy_round")) {                     /* [best,val,nexact] = (A,E,b,tol,it,fun,b_self,mode,screen) */
        /* the loop body of functions/krylov_miobi.m:76-124 in one call: candidate scores + first-wins arg-min (mode 0) /
         * arg-max (mode 1); best is the 1-based row of E (0: none).  screen = -1 reads KR_GREEDY_SCREEN. */
        kr_matrix* M = matrix_of(prhs[0]);
        mwSize nE = mxGetM(prhs[1]);
        int64_t* E = to_i64(prhs[1], NULL);
        int64_t best = -1, info[4] = {0, 0, 0, 0};
        double val = 0.0;
        int screen = (int)mxGetScalar(prhs[8]);
        if (screen < 0) { const char* e = getenv("KR_GREEDY_SCREEN"); screen = (e && atoi(e) != 0) ? 1 : 0; }
        chk(kr_greedy_round(ctx(), M, (int64_t)nE, E, mxGetScalar(prhs[2]), mxGetScalar(prhs[6]), mxGetScalar(prhs[3]),
                            (int64_t)mxGetScalar(prhs[4]), fun_of(prhs[5]), (int)mxGetScalar(prhs[7]), screen, &best, &val,
                            NULL, NULL, info));
        plhs[0] = scalar((double)(best + 1));
        if (nlhs > 1) plhs[1] = scalar(val);
        if (nlhs > 2) plhs[2] = scalar((double)info[0]);
        mxFree(E);
    } else if (!strcmp(op, "fun_update")) {                        /* [Xm,iter,lucky,Um] = (A,U,B,fun,tol,it,want_basis) */
        kr_matrix* M = matrix_of(prhs[0]);
        int64_t dim, it; int lucky, dense;
        mwSize n = mxGetM(prhs[1]);
        int want = (int)mxGetScalar(prhs[6]);
        chk(kr_fun_update(ctx(), M, (int64_t)mxGetN(prhs[1]), mxGetPr(prhs[1]), (int64_t)n, mxGetPr(prhs[2]),
                          (int64_t)mxGetM(prhs[2]), fun_of(prhs[3]), mxGetScalar(prhs[4]), (int64_t)mxGetScalar(prhs[5]),
                          want, &dim, &it, &lucky, &dense));
        plhs[0] = mxCreateDoubleMatrix((mwSize)dim, (mwSize)dim, mxREAL);
        if (nlhs > 3) plhs[3] = mxCreateDoubleMatrix(n, (mwSize)dim, mxREAL);
        chk(kr_fun_update_fetch(ctx(), mxGetPr(plhs[0]), dim, nlhs > 3 ? mxGetPr(plhs[3]) : NULL, (int64_t)n));
        if (nlhs > 1) plhs[1] = scalar((double)it);
        if (nlhs > 2) plhs[2] = mxCreateLogicalScalar(lucky != 0);
    } else if (!strcmp(op, "function_multiple_entries")) {         /* [X,iter] = (A,omega,f,tol,it) */
        kr_matrix* M = matrix_of(prhs[0]);
        mwSize k = mxGetM(prhs[1]);
        int64_t* om = to_i64(prhs[1], NULL);
        int64_t it;
        plhs[0] = mxCreateDoubleMatrix(k, 1, mxREAL);
        chk(kr_function_multiple_entries(ctx(), M, (int64_t)k, om, fun_of(prhs[2]), mxGetScalar(prhs[3]),
                                         (int64_t)mxGetScalar(prhs[4]), mxGetPr(plhs[0]), &it));
        if (nlhs > 1) plhs[1] = scalar((double)it);
        mxFree(om);
    } else if (!strcmp(op, "trace_fun_sparse_update")) {         /* [dtr,q,iter] = (At,Omega,X,fun,tol,it,qmax) */
        kr_matrix* M = matrix_of(prhs[0]);
        mwSize k = mxGetM(prhs[1]);
        int64_t* om = to_i64(prhs[1], NULL);
        int64_t q, it;
        double dtr;
        if (mxGetNumberOfElements(prhs[2]) != k) mexErrMsgTxt("trace_fun_sparse_update: X must have one value per row of Omega");
        chk(kr_trace_fun_sparse_update(ctx(), M, (int64_t)k, om, mxGetPr(prhs[2]), fun_of(prhs[3]), mxGetScalar(prhs[4]),
                                       (int64_t)mxGetScalar(prhs[5]), (int64_t)mxGetScalar(prhs[6]), &dtr, &q, &it, NULL));
        plhs[0] = scalar(dtr);
        if (nlhs > 1) plhs[1] = scalar((double)q);
        if (nlhs > 2) plhs[2] = scalar((double)it);
        mxFree(om);
    } else if (!strcmp(op, "fun_and_grad")) {                      /* [f,gr] = (X,A,Omega,fun,dfun,dfA,tol,it) */
        kr_matrix* M = matrix_of(prhs[1]);
        mwSize k = mxGetM(prhs[2]);
        int64_t* om = to_i64(prhs[2], NULL);
        double f;
        {
            mxArray* gr = mxCreateDoubleMatrix(k, 1, mxREAL);
            chk(kr_fun_and_grad_krylov(ctx(), M, (int64_t)k, mxGetPr(prhs[0]), om, fun_of(prhs[3]), fun_of(prhs[4]),
                                       mxGetPr(prhs[5]), mxGetScalar(prhs[6]), (int64_t)mxGetScalar(prhs[7]), &f, mxGetPr(gr)));
            plhs[0] = scalar(f);
            if (nlhs > 1) plhs[1] = gr; else mxDestroyArray(gr);
        }
        mxFree(om);
    } else if (!strcmp(op, "hessian")) {                           /* Hes = (Atilde, Omega, f, tol, it) */
        kr_matrix* M = matrix_of(prhs[0]);
        mwSize k = mxGetM(prhs[1]);
        int64_t* om = to_i64(prhs[1], NULL);
        int64_t it;
        plhs[0] = mxCreateDoubleMatrix(k, k, mxREAL);
        chk(kr_frechet_hessian(ctx(), M, (int64_t)k, om, fun_of(prhs[2]), mxGetScalar(prhs[3]),
                               (int64_t)mxGetScalar(prhs[4]), mxGetPr(plhs[0]), &it));
        mxFree(om);
    } else if (!strcmp(op, "hessian_multiply")) {      /* [W,iter] = (Atilde, Omega, Y, f, tol, it, reference_form) */
        kr_matrix* M = matrix_of(prhs[0]);
        mwSize k = mxGetM(prhs[1]);
        int64_t* om = to_i64(prhs[1], NULL);
        int64_t it;
        mwSize p = mxGetN(prhs[2]);
        if (mxGetM(prhs[2]) != k) mexErrMsgTxt("hessian_multiply: Y must have one row per row of Omega");
        plhs[0] = mxCreateDoubleMatrix(k, p, mxREAL);
        chk(kr_frechet_hessian_multiply(ctx(), M, (int64_t)k, om, (int64_t)p, mxGetPr(prhs[2]), (int64_t)(k ? k : 1),
                                        fun_of(prhs[3]), mxGetScalar(prhs[6]) != 0.0, mxGetScalar(prhs[4]),
                                        (int64_t)mxGetScalar(prhs[5]), mxGetPr(plhs[0]), (int64_t)(k ? k : 1), &it, NULL));
        if (nlhs > 1) plhs[1] = scalar((double)it);
        mxFree(om);
    } else if (!strcmp(op, "normest")) {                         /* [e,cnt] = (A,tol) */
        double e; int64_t c;
        chk(kr_normest(ctx(), matrix_of(prhs[0]), mxGetScalar(prhs[1]), &e, &c));
        plhs[0] = scalar(e);
        if (nlhs > 1) plhs[1] = scalar((double)c);
    } else if (!strcmp(op, "normAm")) {                            /* [c,mv] = (A,m) */
        double c; int64_t mv;
        chk(kr_normAm(ctx(), matrix_of(prhs[0]), 1.0, (int64_t)mxGetScalar(prhs[1]), &c, &mv));
        plhs[0] = scalar(c);
        if (nlhs > 1) plhs[1] = scalar((double)mv);
    } else if (!strcmp(op, "select_taylor_degree")) {              /* [M,mv,alpha,unA] = (A,ncols,m_max,p_max,shift,force) */
        int64_t mmax = (int64_t)mxGetScalar(prhs[2]), pmax = (int64_t)mxGetScalar(prhs[3]), mv; int unA;
        plhs[0] = mxCreateDoubleMatrix((mwSize)mmax, (mwSize)(pmax - 1), mxREAL);
        { mxArray* al = mxCreateDoubleMatrix((mwSize)(pmax - 1), 1, mxREAL);
          chk(kr_select_taylor_degree(ctx(), matrix_of(prhs[0]), 1.0, (int64_t)mxGetScalar(prhs[1]), mmax, pmax,
                                      (int)mxGetScalar(prhs[4]), (int)mxGetScalar(prhs[5]), mxGetPr(plhs[0]), &mv, mxGetPr(al), &unA));
          if (nlhs > 1) plhs[1] = scalar((double)mv);
          if (nlhs > 2) plhs[2] = al; else mxDestroyArray(al);
          if (nlhs > 3) plhs[3] = scalar((double)unA); }
    } else if (!strcmp(op, "expmv")) {                             /* [f,s,m,mv,mvd,unA] = (t,A,b,M,shift,full_term) */
        kr_matrix* M = matrix_of(prhs[1]);
        mwSize n = mxGetM(prhs[2]), q = mxGetN(prhs[2]);
        int hasM = !mxIsEmpty(prhs[3]);
        int64_t s, m, mv, mvd; int unA;
        plhs[0] = mxCreateDoubleMatrix(n, q, mxREAL);
        chk(kr_expmv(ctx(), M, mxGetScalar(prhs[0]), (int64_t)q, mxGetPr(prhs[2]), (int64_t)n,
                     hasM ? mxGetPr(prhs[3]) : NULL, hasM ? (int64_t)mxGetM(prhs[3]) : 0, hasM ? (int64_t)mxGetN(prhs[3]) : 0,
                     (int)mxGetScalar(prhs[4]), (int)mxGetScalar(prhs[5]), mxGetPr(plhs[0]), (int64_t)n, &s, &m, &mv, &mvd, &unA));
        if (nlhs > 1) plhs[1] = scalar((double)s);
        if (nlhs > 2) plhs[2] = scalar((double)m);
        if (nlhs > 3) plhs[3] = scalar((double)mv);
        if (nlhs > 4) plhs[4] = scalar((double)mvd);
        if (nlhs > 5) plhs[5] = scalar((double)unA);
    } else if (!strcmp(op, "mc_trace")) {                          /* [tr,res,it] = (A,op,tol,maxit,probes) */
        double tr, res; int64_t it;
        chk(kr_mc_trace(ctx(), matrix_of(prhs[0]), (int)mxGetScalar(prhs[1]), mxGetScalar(prhs[2]),
                        (int64_t)mxGetScalar(prhs[3]), mxGetPr(prhs[4]), &tr, &res, &it));
        plhs[0] = scalar(tr);
        if (nlhs > 1) plhs[1] = scalar(res);
        if (nlhs > 2) plhs[2] = scalar((double)it);
    } else if (!strcmp(op, "krylov_start") || !strcmp(op, "krylov_extend") || !strcmp(op, "krylov_free")) {
        /* state handle travels as a uint64 scalar inside params.handle:
         * [V,H,K,last,lucky,handle] = kr_mex('krylov_start', A, b, arnoldi) / ('krylov_extend', handle) */
        kr_krylov* st = NULL; int lucky = 0; int64_t d[5];
        if (!strcmp(op, "krylov_free")) {       /* idempotent: onCleanup of a copied params struct may fire twice */
            kr_krylov* dead = *(kr_krylov**)mxGetData(prhs[0]);
            if (untrack_krylov(dead)) kr_krylov_destroy(dead);
            return;
        }
        if (!strcmp(op, "krylov_start")) {
            chk(kr_krylov_start(ctx(), matrix_of(prhs[0]), (int)mxGetScalar(prhs[2]), (int64_t)mxGetN(prhs[1]),
                                mxGetPr(prhs[1]), (int64_t)mxGetM(prhs[1]), &st, &lucky));
            track_krylov(st);
        } else {
            st = live_krylov(prhs[0]);
            chk(kr_krylov_extend(st, &lucky));
        }
        chk(kr_krylov_dims(st, d));
        /* rows of V = rows of b (start) - the wrapper passes n explicitly on extend as prhs[1] */
        {
            mwSize n = (mwSize)(strcmp(op, "krylov_start") ? mxGetScalar(prhs[1]) : mxGetM(prhs[1]));
            plhs[0] = mxCreateDoubleMatrix(n, (mwSize)d[4], mxREAL);
            plhs[1] = mxCreateDoubleMatrix((mwSize)d[2], (mwSize)d[3], mxREAL);
            plhs[2] = mxCreateDoubleMatrix((mwSize)d[2], (mwSize)d[3], mxREAL);
            plhs[3] = mxCreateDoubleMatrix(n, (mwSize)d[0], mxREAL);
            chk(kr_krylov_get(st, mxGetPr(plhs[0]), (int64_t)n, mxGetPr(plhs[1]), d[2], mxGetPr(plhs[2]), d[2],
                              mxGetPr(plhs[3]), (int64_t)n));
            plhs[4] = mxCreateLogicalScalar(lucky != 0);
            plhs[5] = mxCreateNumericMatrix(1, 1, mxUINT64_CLASS, mxREAL);
            *(kr_krylov**)mxGetData(plhs[5]) = st;
        }
    } else {
        mexErrMsgIdAndTxt("krylov_b200:op", "unknown op '%s'", op);
    }
}
