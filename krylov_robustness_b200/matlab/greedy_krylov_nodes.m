function [nodes, rob_variation, A_new] = greedy_krylov_nodes(A, k, Q, centrality, tol, it, fun)
% Greedy node attack, the node counterpart of functions/greedy_krylov.m: round 1 ranks the nodes by centrality
% (descending, stable) and keeps the top Q+k; every round scores the first Q remaining nodes in ONE device call
% (kr_trace_fun_update_nodes), takes the first-wins arg-min (functions/krylov_miobi.m:112-124), deletes the chosen
% node's off-diagonal entries on the device copy of A and drops the node from the list.
if ~issymmetric(A), error('GREEDY_KRYLOV:: Adjacency matrix should be symmetric'); end
if ~exist('tol', 'var') || isempty(tol), tol = 1e-12; end
if ~exist('it', 'var') || isempty(it), it = min(100, size(A, 1)); end
if ~exist('fun', 'var') || isempty(fun), fun = @exp; end
if ~exist('Q', 'var') || isempty(Q) || Q == 0, Q = full(max(sum(A, 1))); end
[srt, top] = sort(centrality(:), 'descend');
top = top(1:min(Q + k, numel(top)));
nodes = zeros(0, 1); rob_variation = 0;
hA = kr_mex('matrix_create', A);                    % A goes to the device ONCE; the rounds edit it in place
freeA = onCleanup(@() kr_mex('matrix_free', hA));
for r = 1:min(k, numel(top))
    cand = top(1:min(Q, numel(top)));
    vals = kr_mex('trace_fun_update_nodes', hA, double(cand), tol, it, func2str(fun));
    best = 0; bestval = inf;
    for h = 1:numel(vals)
        if vals(h) < bestval, best = h; bestval = vals(h); end
    end
    v = cand(best);
    nb = find(A(:, v));
    nb = nb(nb ~= v);
    if ~isempty(nb)
        A(v, nb) = 0; A(nb, v) = 0;
        kr_mex('matrix_set_edges', hA, v * ones(numel(nb), 1), nb, 0);
    end
    top = top(top ~= v);
    nodes = [nodes; v]; rob_variation = rob_variation + bestval;
end
A_new = A;
end
