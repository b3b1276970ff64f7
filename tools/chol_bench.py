"""Dense Cholesky + explicit inverse micro-benchmark / check (GPU box)."""
import sys, os
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from dbat_b200 import _lib
n = int(sys.argv[1]) if len(sys.argv) > 1 else 2048
rng = np.random.default_rng(0)
M = rng.standard_normal((n, n + 16))
A = M @ M.T + n * np.eye(n)
Ai, ms = _lib.dense_chol_inverse(A, repeat=int(sys.argv[2]) if len(sys.argv) > 2 else 3)
Ar = np.linalg.inv(A)
# useful flops: n^3/3 each for the factor, inv(L) and inv(L)' inv(L)
print('n=%d  factor+inverse %.3f ms  (%.2f TFLOP/s)  inverse rel err %.2e'
      % (n, ms, n ** 3 / ms / 1e9, np.abs(Ai - Ar).max() / np.abs(Ar).max()))
