"""Worst candidates of the 250-candidate break round on a fixture graph: device vs oracle (diagnostic)."""
import sys, warnings, numpy as np
warnings.simplefilter("ignore")
sys.path.insert(0, "."); sys.path.insert(0, "tests")
from conftest import load_graph, edge_UB
import oracle as O
import krylov_robustness_b200 as kr
name = sys.argv[1] if len(sys.argv) > 1 else "misc_Drugs"
A = load_graph(name); n = A.shape[0]
nrm, _ = O.normest(A, 1e-2); tol = 1e-6 * float(np.exp(nrm))
c = O.compute_centrality(A, "eig"); E = O.find_top_edges(A, c, 250, "min")
M = kr.Matrix(A)
x, it, lk = kr.trace_fun_update_edges(M, E, -1.0, tol, 100, "exp")
ox = np.zeros(len(E)); oit = np.zeros(len(E), int)
for h, (i, j) in enumerate(E):
    U, B = edge_UB(n, int(i), int(j), -1.0); ox[h], oit[h], _ = O.trace_fun_update(A, U, B, tol, 100)
rel = np.abs(x - ox) / np.abs(ox)
deg = np.diff(A.indptr)
print(name, "n", n, "tol", tol, "max rel", rel.max(), "iters equal", np.array_equal(it, oit))
for h in np.argsort(-rel)[:8]:
    i, j = E[h]
    print("cand", h, (int(i), int(j)), "deg", deg[i - 1], deg[j - 1], "it", it[h], oit[h], "x", x[h], "ox", ox[h], "rel", rel[h])
    # single call through the general entry point as well
    U, B = edge_UB(n, int(i), int(j), -1.0)
    xs, its, _ = kr.trace_fun_update(M, U, B, tol, 100, 0, "exp")
    print("   single-call path:", xs, its, abs(xs - ox[h]) / abs(ox[h]))
