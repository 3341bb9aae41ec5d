import sys, time, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import krylov_robustness_b200 as kr
from krylov_robustness_b200.graphs import power_law_graph
A = power_law_graph(200_000, 4_000_000, 2.2, seed=3)
A = (A * (1.0 / 64.0)).tocsr()
b = np.random.default_rng(0).standard_normal((A.shape[0], 64))
M = kr.Matrix(A)
V, K, H, p, l = kr.arnoldi_krylov(M, b)
t0 = time.perf_counter()
V, K, H, p, l = kr.arnoldi_krylov(M, b)
for _ in range(4):
    V, K, H, p, l = kr.arnoldi_krylov(V, K, H, p)
dt = time.perf_counter() - t0
print("block arnoldi n=200k bs=64, 5 steps (incl. copying V, H out every call): %.4f s; orth %.2e"
      % (dt, np.linalg.norm(V.T @ V - np.eye(V.shape[1]))))
