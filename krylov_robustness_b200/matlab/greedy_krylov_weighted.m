function [edges, rob_variation, A_new, applied] = greedy_krylov_weighted(A, k, Q, top_edges, tol, it, fun, miobi, weights)
% functions/greedy_krylov.m on a weighted graph, scoring the change each edit makes.  top_edges is the candidate list
% of Q+k rows that functions/greedy_krylov.m:78-83 builds: find_top_edges(A, centrality, Q+k, order) for 'break',
% find_top_missing_edges(A, centrality, Q+k, order) for 'make'.  'break': candidate (i, j) scores B = -A(i, j) *
% [0 1; 1 0], A(i, j) read from the current (edited) A, and the chosen edge is set to 0.  'make': candidate h scores
% B = +weights(h) * [0 1; 1 0] (weights: scalar or aligned with top_edges, default 1) and the chosen pair is set to
% weights(h).  Every round scores the first Q remaining candidates in ONE device call (kr_trace_fun_update_edges_w),
% takes the first-wins extremum (functions/krylov_miobi.m:112-124) and applies exactly the scored change to the
% device copy of A.  applied(r) = A_new(i, j) - A(i, j) of the edge chosen in round r.
if ~issymmetric(A), error('GREEDY_KRYLOV:: Adjacency matrix should be symmetric'); end
if ~exist('tol', 'var') || isempty(tol), tol = 1e-12; end
if ~exist('it', 'var') || isempty(it), it = min(100, size(A, 1)); end
if ~exist('fun', 'var') || isempty(fun), fun = @exp; end
if ~exist('miobi', 'var') || isempty(miobi), miobi = 'break'; end
if ~exist('Q', 'var') || isempty(Q) || Q == 0, Q = full(max(sum(A, 1))); end
make = strcmp(miobi, 'make');
if ~make && ~strcmp(miobi, 'break'), error('KRYLOV_MIOBI:: not supported option for miobi'); end
w = [];
if make
    if ~exist('weights', 'var') || isempty(weights), weights = 1; end
    if isscalar(weights), w = weights * ones(size(top_edges, 1), 1); else, w = weights(:); end
end
edges = zeros(0, 2); rob_variation = 0; applied = zeros(0, 1);
hA = kr_mex('matrix_create', A);                    % A goes to the device ONCE; the rounds edit it in place
freeA = onCleanup(@() kr_mex('matrix_free', hA));
for r = 1:min(k, size(top_edges, 1))
    E = top_edges(1:min(Q, size(top_edges, 1)), :);
    if make
        d = w(1:size(E, 1));
    else
        d = zeros(size(E, 1), 1);
        for h = 1:size(E, 1), d(h) = -full(A(E(h, 1), E(h, 2))); end
    end
    vals = kr_mex('trace_fun_update_edges_w', hA, double(E), d, tol, it, func2str(fun));
    best = 0;
    if make, bestval = -inf; else, bestval = inf; end
    for h = 1:numel(vals)
        if (make && vals(h) > bestval) || (~make && vals(h) < bestval), best = h; bestval = vals(h); end
    end
    i = E(best, 1); j = E(best, 2);
    if make, newval = d(best); else, newval = 0; end
    A(i, j) = newval; A(j, i) = newval;
    kr_mex('matrix_set_edges', hA, i, j, newval);
    keep = ~(top_edges(:, 1) == i & top_edges(:, 2) == j);   % functions/greedy_krylov.m:84-86
    top_edges = top_edges(keep, :);
    if make, w = w(keep); end
    edges = [edges; i j]; rob_variation = rob_variation + bestval; applied = [applied; d(best)];
end
A_new = A;
end
