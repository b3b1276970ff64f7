"""The hot path on projects whose points have a spread of ray counts, up to points seen by every image.

The step picks its point-side kernels by the number of rays of a point: window Schur groups of up to 14 points for
points with up to 20 rays (the wider window instantiation once a group's union exceeds 12 images), the per-point
atomic Schur kernel above 20 rays, and one-thread-per-point assembly and back-substitution (or, with general IO, one
block per point in several passes) above 128 rays.  The scenes here are close-range convergent networks
(synth.make_convergent_scene) whose ray counts sit exactly on those thresholds, and on the limits of a point-side
assembly block (64 points or 128 observations).  Every test first asserts through Problem.reduced_info() that the
handle takes the paths the test exists for, at the production thresholds, then compares with the oracle at the
tolerances of test_gpu_parity.py.
"""
import copy
import functools

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import dbat_b200
from dbat_b200.synth import make_convergent_scene
from oracle import lsa
from oracle.bundle import bundle as obundle, bundle_cov as ocov
from oracle.cameramodel import brown_euler_cam4
from oracle.dbatstruct import buildserialindices, buildweightmatrix, serialize

RES_RTOL = 1e-12
EST_RTOL = 1e-9
EST_ATOL = 1e-11
DENSE_BELOW = 6000          # unknowns: np.linalg.solve of the full normal equations below, the point-first sparse solve above


@pytest.fixture(scope='module', autouse=True)
def _lib(built_lib):
    return built_lib


def dense(a):
    return a.toarray() if hasattr(a, 'toarray') else np.asarray(a)


def relmax(a, b):
    a, b = dense(a), dense(b)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300))


def ray_counts(nOP, nImg, hi, nLong, seed):
    """Rays per point: first a run of 64 two-ray points (a point-side block closed by both of its limits at once),
    then, if hi > 128, a 128-ray point right after a partly filled block (it fills a block alone), then every
    boundary value up to hi four times, then a seeded mix: 2..min(hi, 20) rays with weight 1/(k-1) (many points with
    few rays: they fill window groups of 14) and nLong points with 21..nImg rays."""
    rng = np.random.default_rng(seed)
    head = [2] * 64
    if hi > 128:
        head += [5, 5, 128, 3]
    head += [k for k in (2, 3, 12, 13, 20, 21, 128, 129, nImg) if k <= hi] * 4
    k = np.arange(2, min(hi, 20) + 1)
    w = 1.0 / (k - 1)
    rest = np.concatenate([rng.choice(k, nOP - len(head) - nLong, p=w / w.sum()), rng.integers(21, nImg + 1, nLong)])
    return np.concatenate([head, rng.permutation(rest)])


# mid-size scenes: >= 16 576 estimated points with at most 20 rays, so that the group cap reaches 14 points
SCENES = {
    'spread-small': dict(nImg=160, nOP=20000, hi=12, nLong=0, seed=101),
    'spread-large': dict(nImg=160, nOP=20000, hi=20, nLong=0, seed=102),
    'spread-long': dict(nImg=160, nOP=20000, hi=160, nLong=800, seed=103),
    # small variants of spread-long (dense oracle): fixed points and OP priors, estimated skew (generic evaluation
    # kernels), two IO blocks (general IO kernels)
    'long-fixed': dict(nImg=140, nOP=800, hi=140, nLong=40, seed=104, variant='fixed'),
    'long-skew': dict(nImg=140, nOP=800, hi=140, nLong=40, seed=105, variant='skew'),
    'long-twocam': dict(nImg=140, nOP=800, hi=140, nLong=40, seed=106, variant='two-cameras'),
}


@functools.lru_cache(maxsize=None)
def _scene(name):
    c = SCENES[name]
    rays = ray_counts(c['nOP'], c['nImg'], c['hi'], c['nLong'], c['seed'])
    s, truth = make_convergent_scene(c['nImg'], c['nOP'], rays, seed=c['seed'], build_indices=False)
    assert np.array_equal(np.bincount(s.IP.op, minlength=c['nOP']), rays)
    v = c.get('variant')
    if v == 'fixed':
        big = np.flatnonzero(rays > 128)
        mid = np.flatnonzero((rays > 20) & (rays <= 128))
        sh = np.flatnonzero((rays > 12) & (rays <= 20))
        for j, rows in ((big[0], slice(0, 3)), (big[1], slice(2, 3)), (mid[0], slice(0, 3)), (mid[1], slice(0, 2)),
                        (sh[0], slice(0, 3)), (sh[1], slice(1, 3))):
            s.bundle.est.OP[rows, j] = False                 # fully or partly fixed, at the true position
            s.OP.val[rows, j] = truth['OP'][rows, j]
        s.prior.OP.use[:, big[2]] = True
        s.prior.OP.val[:, big[2]] = truth['OP'][:, big[2]]
        s.prior.OP.std[:, big[2]] = 0.01
    elif v == 'skew':
        s.bundle.est.IO[4, :] = True
    elif v == 'two-cameras':
        cam = (np.arange(c['nImg']) % 2) + 1
        s.IO.struct.block[:] = cam[None, :]
        s.IO.val[0, cam == 2] *= 1.01
        s.IO.val[1, cam == 2] += 0.05
    buildserialindices(s)
    return s, rays


def scene(name):
    s, rays = _scene(name)
    return copy.deepcopy(s), rays


@functools.lru_cache(maxsize=None)
def _oracle(name):
    """Residual, Jacobian and the weighted normal equations of the oracle at the start values."""
    s, _ = _scene(name)
    x0 = serialize(s)
    ro, Jo = brown_euler_cam4(x0, s, True)
    R = np.sqrt(buildweightmatrix(s))
    Jw = Jo.multiply(R[:, None]).tocsc()
    Jw.sort_indices()
    rw = ro * R
    return x0, ro, Jo.tocsc(), Jw, rw, (Jw.T @ Jw).tocsc()


def oracle_step(name, lam):
    s, _ = _scene(name)
    x0, _, _, Jw, rw, N = _oracle(name)
    n = len(x0)
    if n < DENSE_BELOW:
        return np.linalg.solve(N.toarray() + lam * np.eye(n), -(Jw.T @ rw))
    import scipy.sparse as sp
    return lsa.solve_spd_pointfirst(N + lam * sp.identity(n, format='csc'), -(Jw.T @ rw), n - len(s.bundle.serial.OP.dest))


def check_paths(name, info):
    """The handle takes the point-side paths the scene exists for (Problem.reduced_info, slots 12-15)."""
    s, rays = _scene(name)
    est = s.bundle.est.OP.any(axis=0)
    assert info['nPsbig'] == np.count_nonzero(rays > 128)
    assert info['nBig'] == np.count_nonzero(est & (rays > 20))
    if name == 'spread-small':
        assert info['grpMaxRays'] <= 12 and info['grpMaxPts'] == 14 and info['nBig'] == info['nPsbig'] == 0
    elif name == 'spread-large':
        assert 12 < info['grpMaxRays'] <= 20 and info['grpMaxPts'] == 14 and info['nBig'] == info['nPsbig'] == 0
    elif name == 'spread-long':
        assert 12 < info['grpMaxRays'] <= 20 and info['grpMaxPts'] == 14 and info['nBig'] > 0 and info['nPsbig'] > 0
    else:
        assert info['nBig'] > 0 and info['nPsbig'] > 0


@pytest.mark.parametrize('name', list(SCENES))
def test_residual_and_jacobian(name):
    s, _ = scene(name)
    x0, ro, Jo, Jw, _, _ = _oracle(name)
    P = dbat_b200.Problem(s)
    check_paths(name, P.reduced_info())
    r = P(x0)
    assert r.shape == ro.shape and relmax(r, ro) < RES_RTOL
    for weighted, Jref in ((False, Jo), (True, Jw)):
        J = P.jacobian(weighted)
        Jref = Jref.copy()
        Jref.sort_indices()
        assert J.shape == Jref.shape
        assert np.array_equal(J.indptr, Jref.indptr), 'column pointers differ'
        assert np.array_equal(J.indices, Jref.indices), 'row indices differ'
        np.testing.assert_allclose(J.data, Jref.data, rtol=1e-11, atol=1e-13 * np.abs(Jref.data).max())
    P.close()


@pytest.mark.parametrize('name', list(SCENES))
def test_damped_step(name):
    """Schur + Cholesky step against the oracle's solve of the full normal equations (J'J + lambda I) p = -J'r at
    (lambda, Jacobi) = (0, off), (1e3, off), (0, on), with f, |Jp|^2 and r'Jp.  A second step on the same handle is
    bit-identical where every point has at most 20 rays; with more, k_schur_atomic adds in no fixed order and the
    second step only has to meet the same tolerances."""
    s, rays = scene(name)
    x0, _, _, Jw, rw, _ = _oracle(name)
    P = dbat_b200.Problem(s)
    check_paths(name, P.reduced_info())
    deterministic = rays.max() <= 20
    for lam, jacobi in ((0.0, False), (1e3, False), (0.0, True)):
        po = oracle_step(name, lam)
        jp = Jw @ po
        p, st = P.normal_step(x0, lam, jacobi)
        p2, st2 = P.normal_step(x0, lam, jacobi)
        if deterministic:
            assert np.array_equal(p, p2), 'not bit-reproducible'
        for q, t in ((p, st), (p2, st2)):
            assert relmax(q, po) < 5e-9, (lam, jacobi)
            assert abs(t['f'] - 0.5 * rw @ rw) <= 1e-12 * 0.5 * rw @ rw
            assert abs(t['jp2'] - jp @ jp) <= 1e-9 * (jp @ jp)
            assert abs(t['rjp'] - rw @ jp) <= 1e-9 * abs(rw @ jp)
    P.close()


def test_gna_spread_long():
    """A complete GNA run on spread-long against the oracle's: iteration count, first and last residual norm,
    sigma0, estimates.  The residual norms in between are left out: on this network the oracle's GNA solve (SuperLU
    on the column-scaled normal matrix) is itself 1.1e-8 away from its point-first Cholesky of the same system, and
    the residual norm after the first step differs by 4e-9 between the two.  The device's step is held to the
    point-first solve at 5e-9 in test_damped_step; both runs end on the same minimum."""
    s, _ = scene('spread-long')
    s1, s2 = copy.deepcopy(s), copy.deepcopy(s)
    s1, ok, it, s0, E = dbat_b200.bundle(s1, 'gna')
    n, nOPx = len(E.x), len(s.bundle.serial.OP.dest)
    lsa.set_ordering(np.concatenate([np.arange(n - nOPx, n), np.arange(n - nOPx)[::-1]]))     # [OP; EO; IO], as bundle_cov.m:73-84
    try:
        s2, oko, ito, s0o, Eo = obundle(s2, 'gna')
    finally:
        lsa.set_ordering(None)
    assert ok and oko and it == ito
    np.testing.assert_allclose(E.res[[0, -1]], Eo.res[[0, -1]], rtol=1e-12)
    np.testing.assert_allclose(s0, s0o, rtol=EST_RTOL)
    np.testing.assert_allclose(E.x, Eo.x, rtol=EST_RTOL, atol=EST_ATOL)


def test_covariances_with_fixed_long_points():
    """long-fixed after GNA: posterior covariances (bundle_cov) and the device's standard deviations (cov_stats)
    against the oracle's, with fully and partly fixed points of 13-20, 21-128 and 129+ rays and OP priors on a
    129+ ray point."""
    s, _ = scene('long-fixed')
    s1, s2 = copy.deepcopy(s), copy.deepcopy(s)
    s1, ok, it, s0, E = dbat_b200.bundle(s1, 'gna')
    s2, oko, ito, s0o, Eo = obundle(s2, 'gna')
    assert ok and oko and it == ito
    np.testing.assert_allclose(s0, s0o, rtol=EST_RTOL)
    np.testing.assert_allclose(E.x, Eo.x, rtol=EST_RTOL, atol=EST_ATOL)
    for w in ('CIO', 'CEO', 'COP', 'CXX'):
        Cg, Co = dense(dbat_b200.bundle_cov(s1, E, w)), dense(ocov(s2, Eo, w))
        assert Cg.shape == Co.shape and relmax(Cg, Co) < 1e-8, w
    st = E.problem.cov_stats(s0, 0.3)
    assert not st['failed']
    Cxx = dense(ocov(s2, Eo, 'CXX'))
    np.testing.assert_allclose(st['std'], np.sqrt(np.diag(Cxx)), rtol=1e-6)
    E.problem.close()
