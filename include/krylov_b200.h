/*
 * krylov_b200.h - C ABI of libkrylov_b200.so: the B200 (sm_100a) engine behind the MATLAB function
 * signatures of COMPiLELab/krylov_robustness' Krylov matrix-function path.
 *
 * Every entry point names the reference interface it replaces (file:line under the reference
 * tree).  Conventions at this boundary (SURVEY.md 8b):
 *   - plain pointers and sizes only; all pointers are HOST pointers unless the name ends in _dev;
 *   - dense blocks are column-major fp64 (MATLAB layout) with an explicit leading dimension;
 *   - sparse A is CSR (row_ptr[n+1], col_idx[nnz], val[nnz]), 0-based, int64 indices.  MATLAB's CSC
 *     arrays (Jc, Ir, Pr) of a symmetric matrix ARE its CSR arrays and can be passed unchanged;
 *   - node / edge index lists (omega, E) are int64 and 1-BASED, as in the reference;
 *   - every function returns 0 on success, a negative kr_status otherwise, and kr_last_error()
 *     returns the message of the last failure on the calling thread.  There is no CPU fallback:
 *     a missing/failed GPU is KR_ERR_CUDA.
 *   - the library never keeps a host pointer after a call returns; outputs go into caller buffers.
 */
#ifndef KRYLOV_B200_H
#define KRYLOV_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct kr_ctx kr_ctx;         /* one per GPU: stream, library handles, scratch arena      */
typedef struct kr_matrix kr_matrix;   /* device-resident CSR of A (+ transpose when unsymmetric)  */
typedef struct kr_dense kr_dense;     /* device-resident n x k fp64 block (panel-major)           */
typedef struct kr_krylov kr_krylov;   /* device-resident block Lanczos / Arnoldi state (params)   */

enum kr_status {
    KR_OK = 0,
    KR_ERR_ARG = -1,        /* bad argument (message carries the reference's error string)        */
    KR_ERR_CUDA = -2,       /* CUDA / cuBLAS / cuSOLVER failure, or no device                     */
    KR_ERR_NOMEM = -3,
    KR_ERR_UNSUPPORTED = -4
};

/* f selectors: the reference compares handles with isequal(f,@exp) etc.
 * (functions/trace_fun_update.m:43, functions/fun_update.m:43-59). */
enum kr_fun { KR_FUN_EXP = 0, KR_FUN_SINH = 1, KR_FUN_COSH = 2 };

const char* kr_last_error(void);
const char* kr_version(void);

/* ------------------------------------------------------------------ context / matrices / blocks */
int  kr_ctx_create(int device, kr_ctx** out);
void kr_ctx_destroy(kr_ctx* ctx);
int  kr_ctx_sync(kr_ctx* ctx);
/* counters since creation: [0] kernel launches of this library, [1] SpMM launches,
 * [2] matrix-vector products (an n x k SpMM counts k), [3] H2D bytes, [4] D2H bytes */
int  kr_ctx_counters(kr_ctx* ctx, int64_t out[5]);
/* CUDA-event time (ms) accumulated in SpMM kernels since the last call with reset != 0.
 * Only measured while kr_ctx_set_timing(ctx, 1) is on (adds two event records per SpMM). */
int  kr_ctx_set_timing(kr_ctx* ctx, int on);
int  kr_ctx_spmm_time(kr_ctx* ctx, int reset, double* ms, int64_t* launches);
void* kr_ctx_stream(kr_ctx* ctx);     /* cudaStream_t the library launches on */

/* Replaces MATLAB's sparse A as used at functions/lanczos_krylov.m:81, arnoldi_krylov.m:86,
 * expmv.m:77, normAm.m:20.  Values that are all equal are stored pattern-only (4 B / nonzero). */
int  kr_matrix_create(kr_ctx* ctx, int64_t n, int64_t nnz, const int64_t* row_ptr,
                      const int64_t* col_idx, const double* val, kr_matrix** out);
void kr_matrix_destroy(kr_matrix* A);
/* n, nnz, symmetric and nonnegative describe A with every kr_matrix_set_edges edit applied, pending or folded;
 * asking folds nothing in.  pattern_only describes the storage: set when every stored value is the same number,
 * and it keeps describing the stored CSR while edits are pending. */
int  kr_matrix_info(const kr_matrix* A, int64_t* n, int64_t* nnz, int* symmetric, int* pattern_only,
                    int* nonnegative);
/* A(i,j) = A(j,i) = v for count 1-based pairs; v = 0 deletes the entry
 * (functions/krylov_miobi.m:127-135). */
int  kr_matrix_set_edges(kr_matrix* A, int64_t count, const int64_t* i, const int64_t* j, const double* v);

/* Multi-GPU inside ONE process (SURVEY.md 8e: A replicated - it fits 180 GB many times over - and the independent
 * units of the path split across GPUs with one exchange of scalars).  Puts a replica of A, with a context and stream
 * of its own, on each listed device (ndev <= 0 or devices == NULL: the first |ndev| / all visible devices).
 * Afterwards kr_trace_fun_update_edges(_ex) splits its candidate edges and kr_slq_trace(_sign) its probe columns
 * contiguously across the replicas, one host thread per GPU, results gathered in the caller's buffers
 * (functions/krylov_miobi.m:76-124: candidate loop + arg-min over all scores; trace partials summed in a fixed
 * order); kr_matrix_set_edges edits every replica.  Environment KR_GPUS=N makes kr_matrix_create do this itself, so
 * that callers that know nothing about devices - the MATLAB wrappers, Tests/<name>.m unchanged - use N GPUs. */
int  kr_matrix_replicate(kr_matrix* A, int ndev, const int* devices);
int  kr_matrix_replicas(const kr_matrix* A);          /* 1 + number of replicas */

int  kr_dense_create(kr_ctx* ctx, int64_t n, int64_t k, kr_dense** out);
void kr_dense_destroy(kr_dense* d);
int  kr_dense_upload(kr_dense* d, const double* host, int64_t ld);     /* col-major host -> device */
int  kr_dense_download(const kr_dense* d, double* host, int64_t ld);
/* fill with the counter-based Rademacher stream sign(splitmix64(seed, i, j)) (bench / tests) */
int  kr_dense_fill_rademacher(kr_dense* d, uint64_t seed, int64_t col_offset);

/* ------------------------------------------------------------------ L0: operator application */
/* Y = A * X, X n x k col-major.  Replaces `A*w` (functions/lanczos_krylov.m:81). */
int  kr_spmm(kr_ctx* ctx, const kr_matrix* A, int64_t k, const double* X, int64_t ldx,
             double* Y, int64_t ldy);
int  kr_spmm_dev(kr_ctx* ctx, const kr_matrix* A, const kr_dense* X, kr_dense* Y);

/* ------------------------------------------------------------------ L1: Krylov basis builders */
/* [V,H,params,lucky] = lanczos_krylov(A,b)        functions/lanczos_krylov.m:30-58
 * [V,K,H,params,lucky] = arnoldi_krylov(A,b)      functions/arnoldi_krylov.m:32-62
 * arnoldi != 0 selects the Arnoldi variant.  The returned handle is `params` (+V, H, K). */
int  kr_krylov_start(kr_ctx* ctx, const kr_matrix* A, int arnoldi, int64_t bs, const double* b,
                     int64_t ldb, kr_krylov** out, int* lucky);
/* lanczos_krylov(V,H,params) / arnoldi_krylov(V,K,H,params): one more add_inf_pole
 * (functions/lanczos_krylov.m:60-67, functions/arnoldi_krylov.m:64-72). */
int  kr_krylov_extend(kr_krylov* st, int* lucky);
/* sizes: bs, steps j, rows of H ((j+1)*bs), cols of H (j*bs), cols of V (2*bs Lanczos window or
 * (j+1)*bs for Arnoldi) */
int  kr_krylov_dims(const kr_krylov* st, int64_t dims[5]);
/* copy out V (n x vcols), H (hrows x hcols), K (Arnoldi only; may be NULL), params.last (n x bs) */
int  kr_krylov_get(const kr_krylov* st, double* V, int64_t ldv, double* H, int64_t ldh,
                   double* K, int64_t ldk, double* last, int64_t ldl);
void kr_krylov_destroy(kr_krylov* st);

/* ------------------------------------------------------------------ L2: evaluators */
/* [Xm,iter,lucky] = trace_fun_update(A,U,B,tol,it,debug,fun)   functions/trace_fun_update.m:1-130 */
int  kr_trace_fun_update(kr_ctx* ctx, const kr_matrix* A, int64_t rk, const double* U, int64_t ldu,
                         const double* B, int64_t ldb, double tol, int64_t it, int fun,
                         double* Xm, int64_t* iter, int* lucky);
/* The candidate loop of functions/krylov_miobi.m:76-99, all candidates at once: for every edge
 * E(h,:) (1-based, nE x 2 column-major) U = [e_i e_j], B = b_offdiag * [0 1; 1 0]
 * (rank one, B = b_offdiag, when i == j).  Outputs one trace_fun_update result per candidate. */
int  kr_trace_fun_update_edges(kr_ctx* ctx, const kr_matrix* A, int64_t nE, const int64_t* E,
                               double b_offdiag, double tol, int64_t it, int fun,
                               double* Xm, int64_t* iter, int* lucky);
/* Same with the rank-one value given separately: the reference does NOT divide the self-loop update by
 * `rescale` (functions/krylov_miobi.m:88-94: B = -1 / B = 1), only the rank-two one (:78-80). */
int  kr_trace_fun_update_edges_ex(kr_ctx* ctx, const kr_matrix* A, int64_t nE, const int64_t* E,
                                  double b_offdiag, double b_self, double tol, int64_t it, int fun,
                                  double* Xm, int64_t* iter, int* lucky);
/* Node removal, scored for every candidate node V[h] (1-based, nV of them): Xm[h] = tr f(Ã) - tr f(A), where Ã is A
 * with the off-diagonal entries of row and column v set to zero (a_vv kept, n unchanged).  This is
 * trace_fun_update(A, U, B) with U = [e_v, a'], a' the off-diagonal part of row v, B = -[0 1; 1 0]
 * (functions/trace_fun_update.m:72-124), restated without its rank-deficient block: range(U) lies in K_2(A, e_v), so
 * K_j(A, U) = K_{j+1}(A, e_v) and step j is a single-vector Lanczos run from e_v (functions/lanczos_krylov.m:73-101,
 * bs = 1, three-term recurrence): Gm = T_{j+1}, tGm = Gm with its (1,2) and (2,1) entries zeroed, Xm = the trace
 * formula of :83-89 on sort(eig(tGm)), sort(eig(Gm)); stop by the lag-2 rule (:104-118) or when beta_{j+1} < 1e-8
 * (:119-124, lucky).  iter[h] = j at the stop (at most it, 1 <= it <= 128).  A node with no off-diagonal entry scores
 * 0 with iter 1, lucky.  Pending kr_matrix_set_edges edits count, those of v's own row included.  A must be symmetric
 * (the reference's message otherwise).  With replicas (kr_matrix_replicate) the candidates are split contiguously
 * across the GPUs as in kr_trace_fun_update_edges_ex; results are bit-identical run to run and across replicas. */
int  kr_trace_fun_update_nodes(kr_ctx* ctx, const kr_matrix* A, int64_t nV, const int64_t* V, double tol, int64_t it,
                               int fun, double* Xm, int64_t* iter, int* lucky);
/* One round of the greedy loop, functions/krylov_miobi.m:76-124: score every candidate edge (as
 * kr_trace_fun_update_edges_ex) and select arg-min (mode 0, 'break') / arg-max (mode 1, 'make') with the reference's
 * strict first-wins comparison (:112-124).  best = 0-based index into E (-1: none), best_val = its value.
 * screen != 0: when the candidates are dense in few nodes (find_top_missing_edges(...,'min'): 10^5 candidates on ~520
 * nodes) shared per-node Krylov bases rule out the candidates that cannot win (csrc/nodepairs.cuh: values to
 * 1e-9..1e-8 relative, NOT the 1e-10 parity path) and only the contenders - within 1e-6 relative of the approximate
 * leader, plus everything the screen could not settle - are scored by the exact path; the selection runs on exact
 * values, so best / best_val equal those of screen == 0.  scores (nE, may be NULL): exact values where exact[h] != 0,
 * screen values elsewhere.  info (may be NULL): {exactly scored, screened, distinct nodes, basis levels}. */
int  kr_greedy_round(kr_ctx* ctx, const kr_matrix* A, int64_t nE, const int64_t* E, double b_offdiag, double b_self,
                     double tol, int64_t it, int fun, int mode, int screen, int64_t* best, double* best_val,
                     double* scores, int* exact, int64_t* info);
/* Candidate loop of functions/krylov_miobi.m:76-99 with a value per candidate: for row h = (i, j) of E (1-based,
 * nE x 2 col-major) U = [e_i e_j], B = d[h] * [0 1; 1 0]; a self loop i == j is the rank-one update B = d[h].
 * Everything else as kr_trace_fun_update_edges_ex (tol, it, fun, lag-2 / lucky stops of functions/trace_fun_update.m:
 * 104-124, pending edits, replicas: d is split with E).  d[h] = -w removes an edge of weight w, d[h] = +w adds one;
 * d[h] == 0 is scored like any other value (Xm = 0).  With d[h] == b_offdiag for every non-self-loop row and
 * d[h] == b_self for every self loop the outputs are bitwise those of kr_trace_fun_update_edges_ex.  Errors: null d
 * with nE > 0, a non-finite d[h], an index out of range, it < 1, an unsupported fun. */
int  kr_trace_fun_update_edges_w(kr_ctx* ctx, const kr_matrix* A, int64_t nE, const int64_t* E, const double* d,
                                 double tol, int64_t it, int fun, double* Xm, int64_t* iter, int* lucky);
/* kr_greedy_round with a value per candidate (B = d[h] * [0 1; 1 0], as kr_trace_fun_update_edges_w): same screen,
 * same margins and safety net, same first-wins selection (functions/krylov_miobi.m:112-124) on exact values. */
int  kr_greedy_round_w(kr_ctx* ctx, const kr_matrix* A, int64_t nE, const int64_t* E, const double* d, double tol,
                       int64_t it, int fun, int mode, int screen, int64_t* best, double* best_val, double* scores,
                       int* exact, int64_t* info);
/* [Xm,iter,lucky,Um] = fun_update(A,U,B,fun,tol,it,debug)       functions/fun_update.m:1-137
 * want_basis stands in for nargout == 4 (:69,:77).  Xm is returned column-major with leading
 * dimension xm_dim; Um (n x xm_dim, or the Lanczos window) only if want_basis.  Call with
 * Xm == NULL to run and query sizes, then kr_fun_update_fetch. */
int  kr_fun_update(kr_ctx* ctx, const kr_matrix* A, int64_t rk, const double* U, int64_t ldu,
                   const double* B, int64_t ldb, int fun, double tol, int64_t it, int want_basis,
                   int64_t* xm_dim, int64_t* iter, int* lucky, int* dense_fallback);
int  kr_fun_update_fetch(kr_ctx* ctx, double* Xm, int64_t ldx, double* Um, int64_t ldum);
/* [X,iter] = function_multiple_entries(A,omega,f,tol,it,poles,debug)
 * functions/function_multiple_entries.m:1-172 (poles = inf only, :92). omega k x 2 col-major.
 * One single-vector Arnoldi space per distinct first index (:42, :86-110).  On a symmetric matrix a space whose vectors stay
 * on a small ball around its start node (road networks) is run whole by one CTA in shared memory (csrc/entries_local.cuh);
 * the others are advanced together by n x R SpMMs.  Same arithmetic (arnoldi_krylov.m:104-106), same iteration count.
 * Environment (testing): KR_ENTRIES_LOCAL=0 dense batch only, KR_ENTRIES_CHUNK_COLS=c columns per dense chunk. */
int  kr_function_multiple_entries(kr_ctx* ctx, const kr_matrix* A, int64_t k, const int64_t* omega,
                                  int fun, double tol, int64_t it, double* X, int64_t* iter);
/* Objective of the all-edges callback (functions/fun_and_grad_krylov_fun.m:65 with Omega = all edges) without two
 * large traces that cancel: dtr = tr f(Atilde) - tr f(Atilde - D), where D = Delta(X, Omega) is the symmetric sparse matrix
 * with D(i,j) = D(j,i) = X[h] for every row (i, j) of Omega (nomega x 2 col-major, 1-based; duplicates add up, a diagonal
 * pair gives D(i,i) = X[h]).  With A_t = Atilde - (1 - t) D, dtr = int_0^1 sum_h c_h X_h f'(A_t)(i_h, j_h) dt (c_h = 2 off
 * the diagonal, 1 on it; f' = exp / cosh / sinh for exp / sinh / cosh) by q-point Gauss-Legendre, each node one set of
 * entries as in kr_function_multiple_entries (same tol and it, same local / dense paths; the local path runs every
 * (start node, quadrature node) pair in one launch per budget tier).  q is the smallest order whose error bound
 * (q!)^4 / ((2q+1) ((2q)!)^3) n ||D||^{2q} e^{||Atilde|| + ||D||} (||D|| <= its inf-norm, ||Atilde|| by normest) is at
 * most tol * sum_h c_h |X_h|, capped at min(qmax, 32); q_used reports it, iter the largest step count of any entry.
 * X = 0 gives exactly 0 with q_used = 0.  Atilde must be symmetric (the reference's message otherwise); pending
 * kr_matrix_set_edges edits are folded in first.  The entries stay on the device and are reduced in a fixed order:
 * results are bit-identical run to run.  info (may be NULL): {columns run by local tiers 1, 2, 3, columns through the
 * dense batch}, a column being one (start node, quadrature node) pair. */
int  kr_trace_fun_sparse_update(kr_ctx* ctx, const kr_matrix* Atilde, int64_t nomega, const int64_t* Omega,
                                const double* X, int fun, double tol, int64_t it, int64_t qmax, double* dtr,
                                int64_t* q_used, int64_t* iter, int64_t* info);
/* [f,gr] = fun_and_grad_krylov_exp(X,A,Omega,eA,tol,it,debug)   functions/fun_and_grad_krylov_exp.m:1-113
 * [f,gr] = fun_and_grad_krylov_fun(X,A,Omega,fun,dfun,dfA,...)  functions/fun_and_grad_krylov_fun.m:1-71
 * fun == dfun == KR_FUN_EXP reproduces the _exp variant (value and gradient from one fun_update). */
int  kr_fun_and_grad_krylov(kr_ctx* ctx, const kr_matrix* A, int64_t nomega, const double* X,
                            const int64_t* Omega, int fun, int dfun, const double* dfA,
                            double tol, int64_t it, double* f, double* gr);
/* Hes = hessianfcn_exp(X,A,Omega,tol,it)        functions/hessianfcn_exp.m:1-17
 * Hes = hessianfcn_fun(X,A,Omega,f,tol,it)      functions/hessianfcn_fun.m:1-17
 * over functions/multiple_frechet_eval.m:1-211.  Atilde = A + Delta(X,Omega) is assembled by the caller
 * (hessianfcn_exp.m:4-7); Hes is nomega x nomega column-major; it is capped at 64 Krylov steps. */
int  kr_frechet_hessian(kr_ctx* ctx, const kr_matrix* Atilde, int64_t nomega, const int64_t* Omega,
                        int fun, double tol, int64_t it, double* Hes, int64_t* iter);
/* W = Hes * Y without assembling Hes: the HessianMultiplyFcn of the all-edges callbacks (functions/hessianfcn_fun.m:1-17
 * over functions/multiple_frechet_eval.m:1-211, Atilde = A + Delta(X,Omega) assembled by the caller).  For every row h =
 * (i, j) of Omega (nomega x 2 col-major, 1-based), U / V are the single-vector Arnoldi bases of K_s(Atilde, e_i) /
 * K_s(Atilde, e_j), X_h the (1,2) block of f([G, e1 e1'; 0, H']) and s the pair's stop step (lag-3 rule, as
 * kr_frechet_hessian; it is capped at 64 steps).  Then W(h, r) = -2 <X_h, U' S_r V>_F with
 *   form 0 (objective): S_r = sum_l Y(l, r) (e_a e_b' + e_b e_a'), (a, b) = Omega(l, :) - the Hessian of
 *                       -(tr f(Atilde) - tr f(A)) when f is the derivative of its function (dfun of the gradient);
 *   form 1 (reference): S_r = sum_l Y(l, r) e_a e_b' - hessianfcn_fun's Hes * Y, except that Hes mirrors row l < h
 *                       from X_l where W uses X_h (the two agree to the Krylov tolerance).
 * Y: nomega x p (ld ldy), W: nomega x p (ld ldw).  Y = 0 gives W = 0 exactly; iter is the largest stop step of any pair.
 * Atilde must be symmetric (the reference's message otherwise); pending kr_matrix_set_edges edits are folded in first.
 * On a graph whose Krylov vectors stay local (road networks) one CTA runs a pair whole on the ball around its two nodes
 * (csrc/hessp_local.cuh, budget tiers up to 24 steps); pairs that outgrow the last tier or need more steps take the dense
 * families of kr_frechet_hessian, in chunks.  Results are bit-identical run to run.  info (may be NULL): {pairs launched
 * on local tiers 1, 2, 3, pairs through the dense families}.  Environment (testing): KR_ENTRIES_LOCAL=0 dense only. */
int  kr_frechet_hessian_multiply(kr_ctx* ctx, const kr_matrix* Atilde, int64_t nomega, const int64_t* Omega,
                                 int64_t p, const double* Y, int64_t ldy, int fun, int form, double tol, int64_t it,
                                 double* W, int64_t ldw, int64_t* iter, int64_t* info);
/* MATLAB normest(A,tol) as used at functions/fun_and_grad_krylov_fun.m:27 */
int  kr_normest(kr_ctx* ctx, const kr_matrix* A, double tol, double* est, int64_t* count);

/* c = compute_centrality(A, type)                   functions/compute_centrality.m:15-17 ('eig'), :20-26 ('pr')
 * kind 0: |leading eigenvector| of A (the reference calls eigs(A,1)); kind 1: PageRank vector, alpha = 0.85.
 * Power iteration on the device (one launch for the reference's graph sizes), unit 2-norm, stop when the
 * iterate moves by less than tol. */
int  kr_compute_centrality(kr_ctx* ctx, const kr_matrix* A, int kind, double tol, int64_t maxit, double* c,
                           int64_t* iters, int* converged);

/* ------------------------------------------------------------------ expmv family */
/* [c,mv] = normAm(A,m)                               functions/normAm.m:1-52
 * scale: the estimate is of ||(scale*A)^m||_1 (expmv passes t*A, functions/expmv.m:41). */
int  kr_normAm(kr_ctx* ctx, const kr_matrix* A, double scale, int64_t m, double* c, int64_t* mv);
/* [M,mv,alpha,unA] = select_taylor_degree(t*A,b,m_max,p_max,prec,shift,bal,force_estm)
 * functions/select_taylor_degree.m:1-68.  M is m_max x (p_max-1) column-major. shift: subtract
 * trace(A)/n first. */
int  kr_select_taylor_degree(kr_ctx* ctx, const kr_matrix* A, double scale, int64_t ncols_b,
                             int64_t m_max, int64_t p_max, int shift, int force_estm,
                             double* M, int64_t* mv, double* alpha, int* unA);
/* [f,s,m,mv,mvd,unA] = expmv(t,A,b,M,prec,shift,bal,full_term,prnt)   functions/expmv.m:1-94
 * M == NULL: select_taylor_degree is run (as expmv.m:39-45); else M is m_max x p_cols. */
int  kr_expmv(kr_ctx* ctx, const kr_matrix* A, double t, int64_t q, const double* b, int64_t ldb,
              const double* M, int64_t m_max, int64_t p_cols, int shift, int full_term,
              double* f, int64_t ldf, int64_t* s, int64_t* m, int64_t* mv, int64_t* mvd, int* unA);
int  kr_theta(double theta[100]);                     /* functions/theta_taylor.mat */

/* ------------------------------------------------------------------ trace estimators */
/* [tr,res,it] = mc_trace(Afun,n,tol,maxit,isAreal,debug)   functions/mc_trace.m:1-62
 * Afun is one of: op = 0 -> @(x) A*x ; op = 1 -> @(x) expmv(1,A,x,[],'double') (trace_exp.m:5).
 * probes: K = ceil(maxit/30) pairs (S_i, G_i), each n x 10 col-major, stored S_1,G_1,S_2,G_2,...
 * (the reference draws them from an unseeded stream, mc_trace.m:43-44). */
int  kr_mc_trace(kr_ctx* ctx, const kr_matrix* A, int op, double tol, int64_t maxit,
                 const double* probes, double* tr, double* res, int64_t* it);
/* Throughput mode (all probes at once; SURVEY.md 8d, config C3): m-step single-vector Lanczos per
 * probe column, estimate mean_z ||z||^2 e1' f(T_z) e1.  vals (k) / alpha, beta (m x k col-major)
 * may be NULL. */
int  kr_slq_trace(kr_ctx* ctx, const kr_matrix* A, int64_t k, const double* Z, int64_t ldz,
                  int64_t m, int fun, double* tr, double* vals, double* alpha, double* beta);
/* Same with Rademacher probes handed over as int8 signs (+1 / -1), column-major with leading dimension ldz:
 * one eighth of the host -> device bytes, expanded to fp64 on the device; the arithmetic is unchanged. */
int  kr_slq_trace_sign(kr_ctx* ctx, const kr_matrix* A, int64_t k, const signed char* Z, int64_t ldz,
                       int64_t m, int fun, double* tr, double* vals, double* alpha, double* beta);
int  kr_slq_trace_dev(kr_ctx* ctx, const kr_matrix* A, const kr_dense* Z, int64_t m, int fun,
                      double* tr, double* vals, double* alpha, double* beta);

#ifdef __cplusplus
}
#endif
#endif
