function [Xm, iter, lucky] = trace_fun_update_nodes(A, V, tol, it, fun)
% Node removal scored for every candidate node V(h) (1-based): Xm(h) = trace(f(At)) - trace(f(A)), At = A with the
% off-diagonal entries of row and column V(h) set to zero.  The reference's trace_fun_update
% (functions/trace_fun_update.m:72-124) with U = [e_v, a'], B = -[0 1; 1 0], run as one single-vector Lanczos per node on
% the B200 through kr_mex -> kr_trace_fun_update_nodes (include/krylov_b200.h); same lag-2 and lucky stops.
if ~exist('tol', 'var') || isempty(tol), tol = 1e-12; end
if ~exist('it', 'var') || isempty(it), it = min(100, size(A, 1)); end
if ~exist('fun', 'var') || isempty(fun), fun = @exp; end
[Xm, iter, lucky] = kr_mex('trace_fun_update_nodes', A, double(V(:)), tol, it, func2str(fun));
end
