"""One fun_and_grad_krylov_fun callback of the weighted experiments (30 modifiable edges) on a small graph: the call
the launch list of scripts/gpu_r02_s.sh is taken from."""
import os
import sys
import time
import warnings

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
warnings.simplefilter("ignore")
import krylov_robustness_b200 as kr  # noqa: E402
import oracle as O  # noqa: E402
from conftest import load_graph  # noqa: E402

name = sys.argv[1] if len(sys.argv) > 1 else "grid_England"
A = load_graph(name)
A = (A / A.max()).tocsr()
n = A.shape[0]
M = kr.Matrix(A)
c = O.compute_centrality(A, "eig")
nrm = float(O.normest(A, 1e-2)[0])
E = O.find_top_edges(A, c, 100, "min")
vals, _ = kr.function_multiple_entries(M, E, "cosh", 1e-6 * float(np.cosh(nrm)), 100)
ind = np.argsort(-vals, kind="stable")[:30]
Om, dfA = E[ind], vals[ind]
x = 0.05 * np.ones(30)
tol = 1e-6 * float(np.sinh(nrm))
kr.fun_and_grad_krylov_fun(x, M, Om, "sinh", "cosh", dfA, tol, 100)
l0 = M.ctx.counters()["launches"]
t0 = time.perf_counter()
f, g = kr.fun_and_grad_krylov_fun(x, M, Om, "sinh", "cosh", dfA, tol, 100)
dt = time.perf_counter() - t0
print("%s: fun_and_grad_krylov_fun (30 edges) %.3f ms, %d launches, f = %.12g" % (name, dt * 1e3, M.ctx.counters()["launches"] - l0, f))
