"""Debug (GPU): the sparse tile Cholesky alone, small to large, each case under a timeout."""
import os, sys, time, signal
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, 'tests'))
import numpy as np
import __graft_entry__ as g
g.build()
from dbat_b200 import _lib
from test_tile_cholesky import _banded_arrow_spd
def alarm(*a): 
    print('TIMEOUT', flush=True); os._exit(3)
signal.signal(signal.SIGALRM, alarm)
for n, bw, border, mode in [(50, 50, 0, 0), (64, 64, 0, 0), (130, 130, 0, 0), (423, 423, 0, 0), (700, 90, 9, 0), (2500, 200, 9, 1), (2500, 200, 9, 2), (6002, 1272, 9, 1), (6002, 1272, 9, 2)]:
    rng = np.random.default_rng(n)
    A = _banded_arrow_spd(n, bw, border, rng)
    b = rng.standard_normal(n)
    signal.alarm(60)
    x, st = _lib.tile_chol_solve(A, b, mode=mode, leaf=40, repeat=5)
    signal.alarm(0)
    ref = np.linalg.solve(A, b)
    err = np.abs(x - ref).max() / np.abs(ref).max()
    print(n, bw, border, mode, 'err %.2e' % err, st, flush=True)
