function [Xm, iter, lucky] = trace_fun_update_edges_w(A, E, d, tol, it, fun)
% The candidate loop of functions/krylov_miobi.m:76-99 with a value per candidate: for row h = (i, j) of E (1-based)
% U = [e_i e_j], B = d(h) * [0 1; 1 0]; a self loop i == j is the rank-one update B = d(h).  d(h) = -A(i, j) scores the
% removal of edge (i, j) with its weight, d(h) = +w the insertion of an edge of weight w.  Each candidate is
% functions/trace_fun_update.m (same lag-2 and lucky stops), all of them in one call on the B200 through kr_mex ->
% kr_trace_fun_update_edges_w (include/krylov_b200.h).  A scalar d applies to every candidate.
if ~exist('tol', 'var') || isempty(tol), tol = 1e-12; end
if ~exist('it', 'var') || isempty(it), it = min(100, size(A, 1)); end
if ~exist('fun', 'var') || isempty(fun), fun = @exp; end
if isscalar(d), d = d * ones(size(E, 1), 1); end
[Xm, iter, lucky] = kr_mex('trace_fun_update_edges_w', A, double(E), double(d(:)), tol, it, func2str(fun));
end
