function [W, iter] = hessp_all_edges(X, A, Omega, f, Y, tol, it, reference_form)
% W = Hes * Y for the all-edges callbacks without assembling Hes.  Atilde = A + XX + XX' as in
% functions/hessianfcn_fun.m:4-7; f is the function whose Frechet derivative is taken (dfun of the gradient).
% By default Hes is the Hessian of the objective -(trace(fun(Atilde)) - trace(fun(A))); reference_form = true gives
% hessianfcn_fun's matrix times Y instead, which leaves out the term of the mirrored direction e_b e_a'.
% kr_mex -> kr_frechet_hessian_multiply (include/krylov_b200.h).  As an fmincon HessianMultiplyFcn, with the objective
% returning X as its Hessian information:
%   opts = optimoptions('fmincon', 'HessianMultiplyFcn', @(X, Y) hessp_all_edges(X, A, Omega, @cosh, Y, tol, it));
if ~exist('tol', 'var') || isempty(tol), tol = 1e-8; end
if ~exist('it', 'var') || isempty(it), it = min(100, size(A, 1)); end
if ~exist('reference_form', 'var') || isempty(reference_form), reference_form = false; end
n = size(A, 1);
XX = sparse(Omega(:, 1), Omega(:, 2), X(:), n, n);
Atilde = A + XX + XX';
[W, iter] = kr_mex('hessian_multiply', Atilde, double(Omega), double(Y), func2str(f), tol, it, double(reference_form));
end
