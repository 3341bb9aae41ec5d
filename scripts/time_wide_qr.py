"""Time of the wide-block path, thin QR included, on a LARGE graph: trace_fun_update with a rank-32 update (an edge set,
Tests/test_unweighted_break.m:94-95 shape) on a power-law graph with n = 200 000."""
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import krylov_robustness_b200 as kr  # noqa: E402
from krylov_robustness_b200.graphs import power_law_graph, spectral_radius_estimate  # noqa: E402

n = 200_000
A = power_law_graph(n, 4_000_000, 2.2, seed=3)
lam = spectral_radius_estimate(A, 30)
A = (A * (1.0 / lam)).tocsr()
M = kr.Matrix(A)
rng = np.random.default_rng(0)
nodes = rng.choice(n, 32, replace=False)
U = np.zeros((n, 32))
U[nodes, np.arange(32)] = 1.0
B = rng.standard_normal((32, 32)) * 0.05
B = 0.5 * (B + B.T)
tol = 1e-8
kr.trace_fun_update(M, U, B, tol, 100)
l0 = M.ctx.counters()["launches"]
t0 = time.perf_counter()
x, it, lucky = kr.trace_fun_update(M, U, B, tol, 100)
dt = time.perf_counter() - t0
print(json.dumps({"n": n, "rk": 32, "ms": dt * 1e3, "steps": int(it),
                  "launches": M.ctx.counters()["launches"] - l0, "Xm": float(x)}))
