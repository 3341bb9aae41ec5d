function [dtr, q, iter] = trace_fun_sparse_update(At, X, Omega, fun, tol, it, qmax)
% dtr = trace(fun(At)) - trace(fun(At - D)), D = Delta(X, Omega): D(i,j) = D(j,i) = X(h) for every row (i, j) of Omega
% (duplicates add up, a diagonal pair gives D(i,i) = X(h)).  The objective of fun_and_grad_krylov_fun
% (functions/fun_and_grad_krylov_fun.m:65) for a large Omega is -trace_fun_sparse_update(A + Delta, X, Omega, fun, ...).
% q-point Gauss-Legendre along At - (1 - t) D, each node one set of entries fun'(A_t)_Omega on the B200 through
% kr_mex -> kr_trace_fun_sparse_update (include/krylov_b200.h); q is chosen from the quadrature's error bound against
% tol * sum_h c_h |X(h)| (c_h = 2 off the diagonal, 1 on it), at most min(qmax, 32); iter is the largest step count.
if ~exist('tol', 'var') || isempty(tol), tol = 1e-12; end
if ~exist('it', 'var') || isempty(it), it = min(100, size(At, 1)); end
if ~exist('qmax', 'var') || isempty(qmax), qmax = 32; end
[dtr, q, iter] = kr_mex('trace_fun_sparse_update', At, double(Omega), double(X(:)), func2str(fun), tol, it, qmax);
end
