"""Bit-reproducible steps and covariances on projects with wide points: estimated points with more than 20 rays, which
the window Schur kernels do not group and schur_wide.cu reduces in a fixed order.

Every GPU test first asserts through Problem.reduced_info() that the handle has wide points, then requires the same
bits from a second call on the same handle and from a second handle (with an unrelated problem run in between), and
the oracle's result at the tolerances of test_ray_spread.py.  The CPU test reads the built library: none of the
kernels the shared-IO Schur path can launch contains an atomic instruction.
"""
import copy
import os
import re
import shutil
import subprocess
import sys

import numpy as np
import pytest
import scipy.sparse as sp

import dbat_b200
from camcal_fixture import camcal_struct
from oracle import lsa
from oracle.bundle import bundle as obundle, bundle_cov as ocov
from oracle.cameramodel import brown_euler_cam4
from oracle.dbatstruct import buildserialindices, buildweightmatrix, serialize
from test_ray_spread import EST_ATOL, EST_RTOL, dense, oracle_step, relmax, scene

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STEP_SCENES = ['camcal', 'spread-long', 'long-fixed', 'long-skew']
STEP_CASES = ((0.0, False), (1e3, False), (0.0, True))


@pytest.fixture(scope='module')
def _lib(built_lib):
    return built_lib


def _struct(name):
    if name == 'camcal':
        s = camcal_struct()
        buildserialindices(s)
        return s
    return scene(name)[0]


def _camcal_step(s, x0, lam):
    """The oracle's point-first solve of (J'J + lam I) p = -J'r on camcal."""
    r, J = brown_euler_cam4(x0, s, True)
    R = np.sqrt(buildweightmatrix(s))
    Jw = (sp.diags(R) @ J).tocsc()
    n = len(x0)
    nC = n - len(s.bundle.serial.OP.dest)
    return lsa.solve_spd_pointfirst((Jw.T @ Jw).tocsc() + lam * sp.identity(n, format='csc'), -(Jw.T @ (R * r)), nC)


def _unrelated():
    """Another problem through the whole step, so that the second handle does not start from the first one's state."""
    s = scene('spread-small')[0]
    P = dbat_b200.Problem(s)
    P.normal_step(serialize(s), 1.0, False)
    P.close()


def _wide(P):
    assert P.reduced_info()['nBig'] > 0


@pytest.mark.gpu
@pytest.mark.parametrize('name', STEP_SCENES)
def test_steps_bit_identical_across_handles(_lib, name):
    s = _struct(name)
    x0 = serialize(s)
    P1 = dbat_b200.Problem(copy.deepcopy(s))
    _wide(P1)
    first = [P1.normal_step(x0, lam, jac) for lam, jac in STEP_CASES]
    again = [P1.normal_step(x0, lam, jac) for lam, jac in STEP_CASES]
    P1.close()
    _unrelated()
    P2 = dbat_b200.Problem(copy.deepcopy(s))
    _wide(P2)
    other = [P2.normal_step(x0, lam, jac) for lam, jac in STEP_CASES]
    P2.close()
    for (lam, jac), (p, st), (p1, st1), (p2, st2) in zip(STEP_CASES, first, again, other):
        for q, t, what in ((p1, st1, 'same handle'), (p2, st2, 'second handle')):
            assert np.array_equal(p, q), (name, lam, jac, what)
            for k in ('f', 'jp2', 'rjp'):
                assert t[k] == st[k], (name, lam, jac, what, k)
        po = _camcal_step(s, x0, lam) if name == 'camcal' else oracle_step(name, lam)
        assert relmax(p, po) < 5e-9, (name, lam, jac)


@pytest.mark.gpu
def test_forced_wide_path_subprocess(_lib):
    """DBAT_GRP_MAXM=6 puts every point of priors+fixed (10 rays each, fixed points and OP priors) on the wide path:
    two handles give the same bits, and the step is the dense oracle's."""
    code = r'''
import sys, copy, numpy as np
sys.path.insert(0, %r); sys.path.insert(0, %r)
import dbat_b200
from test_gpu_parity import scene, CASES
from oracle.cameramodel import brown_euler_cam4
from oracle.dbatstruct import buildweightmatrix, serialize
s, _ = scene(**CASES['priors+fixed'])
x0 = serialize(s); W = buildweightmatrix(s)
steps = []
for h in range(2):
    P = dbat_b200.Problem(copy.deepcopy(s))
    info = P.reduced_info()
    assert info['nBig'] > 0 and info['grpMaxPts'] == 0, info      # no point left for the window kernels
    steps.append(P.normal_step(x0, 10.0, False))
    P.close()
(p1, st1), (p2, st2) = steps
assert np.array_equal(p1, p2) and all(st1[k] == st2[k] for k in ('f', 'jp2', 'rjp'))
ro, Jo = brown_euler_cam4(x0, s, True)
Jw = Jo.multiply(np.sqrt(W)[:, None]).tocsc(); rw = ro * np.sqrt(W)
N = (Jw.T @ Jw).toarray()
po = np.linalg.solve(N + 10.0 * np.eye(N.shape[0]), -(Jw.T @ rw))
assert np.abs(p1 - po).max() / np.abs(po).max() < 5e-9
print('WIDE-OK')
''' % (ROOT, os.path.join(ROOT, 'tests'))
    env = dict(os.environ, DBAT_GRP_MAXM='6')
    out = subprocess.run([sys.executable, '-c', code], env=env, capture_output=True, text=True, timeout=600)
    assert 'WIDE-OK' in out.stdout, out.stdout + out.stderr


@pytest.mark.gpu
@pytest.mark.parametrize('method', ['gna', 'lm'])
@pytest.mark.parametrize('name', ['camcal', 'spread-long'])
def test_optimiser_runs_bit_identical(_lib, name, method):
    s = _struct(name)
    runs = []
    for _ in range(2):
        s1, ok, it, s0, E = dbat_b200.bundle(copy.deepcopy(s), method)
        _wide(E.problem)
        runs.append((ok, it, E.x, E.res, getattr(E.damping, 'alpha' if method == 'gna' else 'lambda')))
        E.problem.close()
    (ok1, it1, x1, res1, d1), (ok2, it2, x2, res2, d2) = runs
    assert ok1 and ok2 and it1 == it2
    assert np.array_equal(x1, x2) and np.array_equal(res1, res2)
    assert np.array_equal(np.asarray(d1), np.asarray(d2))


@pytest.mark.gpu
def test_covariances_bit_identical(_lib):
    """long-fixed after GNA (fully and partly fixed wide points, OP priors on one): bundle_cov CIO / CEO / COP and
    cov_stats twice on each of two handles, bit-identical, and the oracle's covariances at 1e-8."""
    s = scene('long-fixed')[0]
    outs, handles = [], []
    for _ in range(2):
        s1, ok, it, s0, E = dbat_b200.bundle(copy.deepcopy(s), 'gna')
        assert ok
        _wide(E.problem)
        for _rep in range(2):
            C = {w: dense(dbat_b200.bundle_cov(s1, E, w)) for w in ('CIO', 'CEO', 'COP')}
            st = E.problem.cov_stats(s0, 0.3)
            assert not st['failed']
            outs.append((C, st))
        handles.append((s1, E))
        _unrelated()
    C0, st0 = outs[0]
    for C, st in outs[1:]:
        for w in C0:
            assert np.array_equal(C[w], C0[w]), w
        assert np.array_equal(st['std'], st0['std'])
        for k in ('io', 'eo', 'op'):
            for a, b in zip(st[k], st0[k]):
                assert np.array_equal(a, b), k
    s1, E = handles[-1]
    s2, oko, ito, s0o, Eo = obundle(copy.deepcopy(s), 'gna')
    assert oko
    np.testing.assert_allclose(E.x, Eo.x, rtol=EST_RTOL, atol=EST_ATOL)
    for w in C0:
        Co = dense(ocov(s2, Eo, w))
        assert C0[w].shape == Co.shape and relmax(C0[w], Co) < 1e-8, w
    for _, E in handles:
        E.problem.close()


# kernels launch_schur can launch with one shared IO block
SHARED_IO_SCHUR = ('k_build_S', 'k_point_minv', 'k_schur_win', 'k_schur_reduce', 'k_schur_ss_apply', 'k_wide_stage',
                   'k_wide_reduce')


def test_shared_io_schur_kernels_have_no_atomics(_lib):
    cuobjdump = shutil.which('cuobjdump') or '/usr/local/cuda/bin/cuobjdump'
    if not os.path.exists(cuobjdump):
        pytest.skip('cuobjdump not available')
    sass = subprocess.run([cuobjdump, '-sass', _lib], capture_output=True, text=True, check=True).stdout
    funcs = {}
    for part in re.split(r'\n\s*Function : ', sass)[1:]:
        name, body = part.split('\n', 1)
        funcs[name.strip()] = body
    atomic = re.compile(r'\b(ATOM|ATOMG|ATOMS|RED|REDG)\b|\b(ATOMG?S?|REDG?)\.')
    seen = set()
    for mangled, body in funcs.items():
        for k in SHARED_IO_SCHUR:
            if re.search(r'\d%s(I|\d)' % k, mangled):
                seen.add(k)
                assert not atomic.search(body), (k, mangled, atomic.search(body).group(0))
    assert seen == set(SHARED_IO_SCHUR), sorted(set(SHARED_IO_SCHUR) - seen)
    # the pattern does find atomics where they are: the general-IO S assembly keeps them
    gen = [b for m, b in funcs.items() if 'k_build_S_gen' in m]
    assert gen and atomic.search(gen[0])
