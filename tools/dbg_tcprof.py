"""Debug (GPU): per-task time stamps of the tile factorisation -> where the chain time goes."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, 'tests'))
import numpy as np
os.environ['DBAT_TCHOL_PROF'] = os.path.join(ROOT, 'gpurun_out', 'tcprof.csv')
import __graft_entry__ as g
g.build()
from dbat_b200 import _lib
from test_tile_cholesky import _banded_arrow_spd
n, bw, border, mode = 2500, 200, 9, 1
rng = np.random.default_rng(n)
A = _banded_arrow_spd(n, bw, border, rng)
b = rng.standard_normal(n)
x, st = _lib.tile_chol_solve(A, b, mode=mode, leaf=40, repeat=5)
print(st)
import pandas as pd
d = pd.read_csv(os.environ['DBAT_TCHOL_PROF'])
diag = d[d.I == d.J].sort_values('t_end')
print(diag[['I', 'J', 'nterms', 't_claim', 't_terms', 't_deps', 't_end']].head(12).to_string())
print('diag: potrf mean ns', (diag.t_end - diag.t_deps).mean(), 'terms->deps', (diag.t_deps - diag.t_terms).mean())
sub = d[d.I == d.J + 1].sort_values('t_end')
print(sub[['I', 'J', 'nterms', 't_claim', 't_terms', 't_deps', 't_end']].head(12).to_string())
print('subdiag: solve mean ns', (sub.t_end - sub.t_deps).mean(), 'wait+load', (sub.t_deps - sub.t_terms).mean())
# chain: diag end(J) -> subdiag end (J+1,J) -> diag end (J+1)
de = diag.set_index('J').t_end; se = sub.set_index('J').t_end; sd = sub.set_index('J').t_deps; dt = diag.set_index('J').t_terms; dd = diag.set_index('J').t_deps
for J in range(5, 12):
    print(J, 'potrf end', de[J], ' sub deps', sd[J] - de[J], ' sub end', se[J] - de[J], ' next diag terms', dt[J + 1] - de[J], ' deps', dd[J + 1] - de[J], ' end', de[J + 1] - de[J])
