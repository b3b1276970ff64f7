"""CUDA path (through the C ABI) against the CPU oracle and the reference's golden files.

Tolerances are the ones BASELINE.json states: sparsity/indexing bit-exact, residuals rtol
1e-12, final estimates and sigmas rtol 1e-9, identical iteration counts.
"""
import copy
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import dbat_b200
from dbat_b200.synth import make_scene
from camcal_fixture import GOLD, camcal_struct, golden_camera_xml, golden_eo
from oracle import loaders
from oracle.bundle import bundle as obundle, bundle_cov as ocov
from oracle.cameramodel import brown_euler_cam4
from oracle.dbatstruct import buildserialindices, buildweightmatrix, serialize

RES_RTOL = 1e-12
EST_RTOL = 1e-9
# Elements that are (nearly) zero by the choice of the object frame - a point on an axis, an angle of 1e-6 rad -
# have no relative scale; they are held to 1e-11 absolute (the estimates are metres, millimetres and radians: that
# is 1e-9 of a centimetre).  The sum order inside the Schur update is not fixed, so the last bits of such elements
# move by ~1e-12 from run to run.
EST_ATOL = 1e-11


@pytest.fixture(scope='module', autouse=True)
def _lib(built_lib):
    return built_lib


def dense(a):
    """ndarray view of whatever the oracle / product returns (ocov switches to scipy sparse blocks above
    oracle.bundle.BLOCK_PATH_ABOVE unknowns)."""
    return a.toarray() if hasattr(a, 'toarray') else np.asarray(a)


def relmax(a, b):
    a, b = dense(a), dense(b)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300))


def scene(model=3, seed=7, nImg=21, nOP=100, rays=10, priors=False, fixed_pts=0):
    s, truth = make_scene(nImg, nOP, rays=rays, seed=seed, build_indices=False)
    s.IO.model.distModel[:] = model
    if model != 3:           # exercise affine/skew and distortion terms of every model
        s.IO.val[3, :] = 2e-4
        s.IO.val[4, :] = -1e-4 if model >= 3 else 0.0
        s.IO.val[5:10, :] = truth['IO'][5:10, None] * 0.5
        if model in (2, 1, -1):   # setcamest masks aspect/skew for |model|<3 (setcamest.m:46-58)
            s.IO.val[3:5, :] = 0.0
            s.bundle.est.IO[3:5, :] = False
        if model == -1:           # forward model: distortion acts on the ideal point
            s.IO.val[5:10, :] *= -1
    if fixed_pts:
        s.bundle.est.OP[:, :fixed_pts] = False
        s.bundle.est.OP[2, fixed_pts] = False            # one partially fixed point
    if priors:
        s.prior.EO.use[0:3, 3] = True
        s.prior.EO.val[0:3, 3] = truth['EO'][0:3, 3]
        s.prior.EO.std[0:3, 3] = 0.02
        s.prior.OP.use[:, 5:9] = True
        s.prior.OP.val[:, 5:9] = truth['OP'][:, 5:9]
        s.prior.OP.std[:, 5:9] = 0.01
        s.prior.IO.use[0, 0] = True
        s.prior.IO.val[0, 0] = 24.0
        s.prior.IO.std[0, 0] = 0.05
    buildserialindices(s)
    return s, truth


CASES = {
    'model3': dict(model=3),
    'model2': dict(model=2),
    'model4': dict(model=4),
    'model5': dict(model=5),
    'model1': dict(model=1),
    'model-1': dict(model=-1),
    'priors+fixed': dict(model=3, priors=True, fixed_pts=4),
    'ragged': dict(model=3, rays=3, nOP=150, seed=11),
}


@pytest.mark.parametrize('case', list(CASES))
def test_residual_and_jacobian(case):
    s, _ = scene(**CASES[case])
    x0 = serialize(s)
    P = dbat_b200.Problem(copy.deepcopy(s))
    r = P(x0)
    ro, Jo = brown_euler_cam4(x0, s, True)
    assert r.shape == ro.shape
    assert relmax(r, ro) < RES_RTOL
    for weighted in (False, True):
        J = P.jacobian(weighted)
        Jref = Jo if not weighted else Jo.multiply(np.sqrt(buildweightmatrix(s))[:, None]).tocsc()
        Jref.sort_indices()
        assert J.shape == Jref.shape
        assert np.array_equal(J.indptr, Jref.indptr), 'column pointers differ'
        assert np.array_equal(J.indices, Jref.indices), 'row indices differ'
        np.testing.assert_allclose(J.data, Jref.data, rtol=1e-11, atol=1e-13 * np.abs(Jref.data).max())
    P.close()


def test_value_dependent_sparsity_camcal_start():
    """camcal starts with K=P=b=0, so some IO partials are exactly zero and absent from J at the
    first evaluation (multi_res.m `find()`); the pattern must match bit for bit."""
    s = camcal_struct('default', seed=1)
    buildserialindices(s)
    x0 = serialize(s)
    P = dbat_b200.Problem(copy.deepcopy(s))
    r, J = P(x0, True)
    ro, Jo = brown_euler_cam4(x0, s, True)
    assert relmax(r, ro) < RES_RTOL
    assert J.nnz == Jo.nnz and np.array_equal(J.indptr, Jo.indptr) and np.array_equal(J.indices, Jo.indices)
    full = 2 * len(s.IP.img) * (9 + 6) + 0
    assert J.nnz < full + 2 * len(s.IP.img) * 3          # zeros really were dropped
    P.close()


@pytest.mark.parametrize('case', ['model3', 'priors+fixed', 'model5', 'ragged'])
@pytest.mark.parametrize('lam,jacobi', [(0.0, False), (1e3, False), (0.0, True)])
def test_damped_step(case, lam, jacobi):
    """Schur + dense Cholesky step equals the reference's full sparse solve
    p=(J'J+lambda*I)\\(-J'r) (levenberg_marquardt.m:119), and a second step on the same handle is
    bit-identical (the Schur reduction has no atomics for points with up to DBAT_GRP_MAXM rays)."""
    s, _ = scene(**CASES[case])
    x0 = serialize(s)
    W = buildweightmatrix(s)
    P = dbat_b200.Problem(copy.deepcopy(s))
    p, st = P.normal_step(x0, lam, jacobi)
    p2, _ = P.normal_step(x0, lam, jacobi)
    assert np.array_equal(p, p2), 'not bit-reproducible'
    ro, Jo = brown_euler_cam4(x0, s, True)
    Jw = Jo.multiply(np.sqrt(W)[:, None]).tocsc()
    rw = ro * np.sqrt(W)
    N = (Jw.T @ Jw).toarray()
    po = np.linalg.solve(N + lam * np.eye(N.shape[0]), -(Jw.T @ rw))
    assert relmax(p, po) < 5e-9
    assert abs(st['f'] - 0.5 * rw @ rw) <= 1e-12 * 0.5 * rw @ rw
    jp = Jw @ po
    assert abs(st['jp2'] - jp @ jp) <= 1e-9 * (jp @ jp)
    assert abs(st['rjp'] - rw @ jp) <= 1e-9 * abs(rw @ jp)
    P.close()


def _decisions(rr):
    rr = np.asarray(rr)
    return [bool(rr[i + 1] != rr[i]) for i in range(len(rr) - 1)]


@pytest.mark.parametrize('case', ['model3', 'model4', 'model1', 'model-1', 'priors+fixed', 'ragged'])
@pytest.mark.parametrize('damping', ['gna', 'lmp', 'lm'])
def test_optimisers(case, damping):
    s, _ = scene(**CASES[case])
    s1, s2 = copy.deepcopy(s), copy.deepcopy(s)
    s1, ok, it, s0, E = dbat_b200.bundle(s1, damping)
    s2, oko, ito, s0o, Eo = obundle(s2, damping)
    assert E.code == Eo.code == 0
    np.testing.assert_allclose(s0, s0o, rtol=EST_RTOL)
    if damping in ('gna', 'lmp'):
        np.testing.assert_allclose(E.x, Eo.x, rtol=EST_RTOL, atol=EST_ATOL)
        np.testing.assert_allclose(s1.IO.val, s2.IO.val, rtol=EST_RTOL, atol=1e-12)
        np.testing.assert_allclose(s1.EO.val, s2.EO.val, rtol=EST_RTOL, atol=1e-12)
        np.testing.assert_allclose(s1.OP.val, s2.OP.val, rtol=EST_RTOL, atol=1e-12)
        assert it == ito
        np.testing.assert_allclose(E.res, Eo.res, rtol=1e-10)
        np.testing.assert_allclose(E.trace, Eo.trace, rtol=1e-8, atol=1e-10)
    else:
        # LM accepts a trial point iff fNew<f (levenberg_marquardt.m:177).  Once converged that
        # comparison is decided by rounding noise in BOTH implementations (the reference
        # included), so the number of trailing noise-level trials - and with it the last digits
        # of x - may differ; every decision made above the noise floor must be identical and the
        # iterates must agree to 1e-9 up to that point.
        d1, d2 = _decisions(E.res), _decisions(Eo.res)
        k = 0
        while k < min(len(d1), len(d2)) and d1[k] == d2[k]:
            k += 1
        np.testing.assert_allclose(E.res[:k + 1], Eo.res[:k + 1], rtol=1e-10)
        np.testing.assert_allclose(E.trace[:, :k + 1], Eo.trace[:, :k + 1], rtol=EST_RTOL, atol=1e-12)
        if k < min(len(d1), len(d2)):
            a, b = Eo.res[k], (Eo.res[k + 1] if d2[k] else E.res[k + 1])
            assert abs(a - b) <= 1e-9 * a, 'LM decision %d differs above the rounding floor' % k
        else:
            assert it == ito
        np.testing.assert_allclose(E.x, Eo.x, rtol=1e-6, atol=1e-9)
        # ... and whatever the trailing noise-level trials did, both runs sit on the same minimum.  The
        # termination test |Jp| <= 1e-6 |r| (bundle.m:186-192) leaves a step of up to 1e-6 |r| ~ 1e-4 in units of
        # the posterior standard deviations, so that is the meaningful bound per parameter (measured: 2e-6).
        # LM has no golden in the reference ("parity unpinned by the reference", SURVEY §8c): oracle vs CUDA.
        sig = np.sqrt(np.diag(dense(ocov(s2, Eo, 'CXX'))))
        assert np.all(np.abs(E.x - Eo.x) <= 1e-4 * sig), float(np.max(np.abs(E.x - Eo.x) / sig))


def test_mid_size_step_and_solve_against_the_oracle():
    """The 1/10-scale block of BASELINE config 4 (100 cameras x 20 000 points x 200 000 observations, n = 60 602):
    grouped Schur with real group statistics, a dissected and tiled reduced system, multi-chunk images.  One
    damped step against the oracle's sparse solve of the FULL system, then a complete GNA run against the
    oracle's (iteration count, residual norms, estimates)."""
    import scipy.sparse as sp
    from oracle import lsa
    s, _ = make_scene(100, 20000, rays=10, seed=20240607)
    x0 = serialize(s)
    R = np.sqrt(buildweightmatrix(s))
    P = dbat_b200.Problem(copy.deepcopy(s))
    info = P.reduced_info()
    assert info['nT'] >= 9
    ro, Jo = brown_euler_cam4(x0, s, True)
    Jw = (sp.diags(R) @ Jo).tocsc()
    rw = R * ro
    N = (Jw.T @ Jw).tocsc()
    n = len(x0)
    nC = n - len(s.bundle.serial.OP.dest)
    for lam, jacobi in ((0.0, False), (10.0, False), (0.0, True)):
        p, st = P.normal_step(x0, lam, jacobi)
        po = lsa.solve_spd_pointfirst(N + lam * sp.identity(n, format='csc'), -(Jw.T @ rw), nC)
        assert relmax(p, po) < 5e-9, (lam, jacobi)
        jp = Jw @ po
        assert abs(st['f'] - 0.5 * rw @ rw) <= 1e-12 * 0.5 * rw @ rw
        assert abs(st['jp2'] - jp @ jp) <= 1e-9 * (jp @ jp)
        assert abs(st['rjp'] - rw @ jp) <= 1e-9 * abs(rw @ jp)
        # the default path has no atomics anywhere (window Schur + fixed-order sums, data-flow Cholesky with a
        # static term order): the step is bit-identical from run to run
        p2, _ = P.normal_step(x0, lam, jacobi)
        assert np.array_equal(p, p2), 'default path not bit-reproducible'
    P.close()
    s1, s2 = copy.deepcopy(s), copy.deepcopy(s)
    s1, ok, it, s0, E = dbat_b200.bundle(s1, 'gna')
    nOPx = len(s.bundle.serial.OP.dest)
    lsa.set_ordering(np.concatenate([np.arange(n - nOPx, n), np.arange(n - nOPx)[::-1]]))     # [OP; EO; IO], as bundle_cov.m:73-84
    try:
        s2, oko, ito, s0o, Eo = obundle(s2, 'gna')
    finally:
        lsa.set_ordering(None)
    assert ok and oko and it == ito
    # the iterate after the first (large) step agrees to ~2e-9 absolute - two different direct solvers on a system
    # of condition 1e10 - and so does its residual norm to 3e-10; both runs then contract onto the same minimum
    np.testing.assert_allclose(E.res, Eo.res, rtol=1e-9)
    np.testing.assert_allclose(E.res[-1], Eo.res[-1], rtol=1e-12)
    np.testing.assert_allclose(s0, s0o, rtol=EST_RTOL)
    np.testing.assert_allclose(E.x, Eo.x, rtol=EST_RTOL, atol=EST_ATOL)


def test_no_datum_network_is_reported_singular():
    """camcaldemo_no_datum.m on the device: no control points, 7-dimensional gauge freedom.  The reference stops
    with code -2 at iteration 0 (MATLAB's singular-matrix warning; first error 15772.8, sigma0 258.848 in
    camcal-dbatreport-no-datum.txt).  The device's stand-in for that warning is the pivot-ratio test on the
    Jacobi-scaled reduced system (api.cu solve_step); this pins it on the reference's own report."""
    from oracle.loaders import camcal_pm_struct
    G = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'camcalpm')
    s = camcal_pm_struct(os.path.join(G, 'camcal-pmexport.txt'), None, keep_loaded=True)
    so = copy.deepcopy(s)
    s, ok, it, s0, E = dbat_b200.bundle(s, 'gna')
    so, oko, ito, s0o, Eo = obundle(so, 'gna')
    assert not ok and not oko
    assert (E.code, it) == (Eo.code, ito) == (-2, 0) and E.numParams == 435
    assert abs(E.res[0] - 15772.8) < 0.06 and abs(s0 - 258.848) < 6e-4
    np.testing.assert_allclose(s0, s0o, rtol=EST_RTOL)


def test_camcal_golden_end_to_end():
    """CUDA bundle + bundle_cov against the reference's golden files directly."""
    s = camcal_struct('default', seed=1)
    s, ok, iters, s0, E = dbat_b200.bundle(s, 'gna')
    assert ok
    assert abs(s0 - 1.6148) < 5e-5 and abs(E.res[-1] - 98.556) < 5e-4
    gold = loaders.load_camcal_script(GOLD, golden_camera_xml()).IO.val[:, 0]
    np.testing.assert_allclose(s.IO.val[[0, 1, 2], 0], gold[[0, 1, 2]], rtol=2e-8)
    np.testing.assert_allclose(s.IO.val[5:10, 0], gold[5:10], rtol=5e-6)
    _, EOg, stdg = golden_eo()
    np.testing.assert_allclose(s.EO.val, EOg, atol=2e-8)
    CEO = dbat_b200.bundle_cov(s, E, 'CEO')
    sd = np.sqrt(CEO.diagonal()).reshape(6, -1, order='F')
    np.testing.assert_allclose(sd * 180 / np.pi, stdg, rtol=1e-6)
    rows = loaders.load_table(os.path.join(GOLD, 'result', 'top_residuals.txt'))
    idmap = {(int(s.OP.id[j]), int(s.EO.id[i])): k for k, (i, j) in enumerate(zip(s.IP.img, s.IP.op))}
    for r in rows:
        np.testing.assert_allclose(s.post.res.IP[:, idmap[(int(r[0]), int(r[1]))]],
                                   [float(r[4]), float(r[5])], atol=2e-6)


@pytest.mark.parametrize('case', ['model3', 'priors+fixed'])
def test_posterior_covariances(case):
    s, _ = scene(**CASES[case])
    s1, s2 = copy.deepcopy(s), copy.deepcopy(s)
    s1, ok, _, s0, E = dbat_b200.bundle(s1, 'gna')
    s2, oko, _, s0o, Eo = obundle(s2, 'gna')
    assert ok and oko
    for w in ('CIO', 'CEO', 'COP', 'CIOF', 'CEOF', 'COPF', 'CXX'):
        Cg = dbat_b200.bundle_cov(s1, E, w)
        Cg = Cg.toarray() if hasattr(Cg, 'toarray') else Cg
        Co = dense(ocov(s2, Eo, w))
        assert Cg.shape == Co.shape
        assert relmax(Cg, Co) < 1e-8, w
        sg, so = np.sqrt(np.diag(Cg)), np.sqrt(np.diag(Co))
        m = so > 0
        np.testing.assert_allclose(sg[m], so[m], rtol=EST_RTOL * 10)
        assert np.all(sg[~m] == 0)


def test_structural_rank_deficiency_code():
    """A point with a single ray cannot be estimated: code -4 (camcaldemo_1ray golden)."""
    s, _ = scene(model=3)
    k = np.flatnonzero(s.IP.op == 0)
    keep = np.ones(len(s.IP.op), bool)
    keep[k[1:]] = False
    for f in ('val', 'std'):
        setattr(s.IP, f, getattr(s.IP, f)[:, keep])
    for f in ('img', 'op', 'cam'):
        setattr(s.IP, f, getattr(s.IP, f)[keep])
    s.bundle.serial = None
    buildserialindices(s)
    so = copy.deepcopy(s)
    s, ok, _, _, E = dbat_b200.bundle(s, 'gna')
    so, oko, _, _, Eo = obundle(so, 'gna')
    assert E.code == Eo.code == -4 and not ok


def test_unsupported_configurations_fail_loudly():
    s, _ = scene(model=3)
    s.IO.model.distModel[:] = 7
    with pytest.raises(dbat_b200._lib.DbatError):
        dbat_b200.Problem(s)
    s, _ = scene(model=3)                                   # the dense point covariance needs one shared IO block
    s.IO.struct.block[1:3, :] = np.arange(1, s.IO.val.shape[1] + 1)
    s.bundle.serial = None
    buildserialindices(s)
    P = dbat_b200.Problem(s)
    P(serialize(s))
    with pytest.raises(dbat_b200._lib.DbatError):
        P.cov('cxx', 1.0)
    P.close()


def _general_io_scene(kind):
    """IO block structures beyond one shared camera (IO.struct.block, buildserialindices.m:162-221)."""
    s, truth = make_scene(24, 260, rays=8, seed=21, build_indices=False)
    nImg = s.IO.val.shape[1]
    if kind == 'image-variant-pp':
        # romabundledemo_imagevariant.m:44: every image its own principal point, everything else shared
        s.IO.struct.block[1:3, :] = np.arange(1, nImg + 1)
    elif kind == 'two-cameras':
        # setdbatcamsandimages.m:28: one block per camera; the second camera has its own lens
        cam = (np.arange(nImg) % 2) + 1
        s.IO.struct.block[:] = cam[None, :]
        s.IO.val[0, cam == 2] *= 1.01
        s.IO.val[1, cam == 2] += 0.05
    elif kind == 'image-variant-all':
        s.IO.struct.block[:] = np.arange(1, nImg + 1)[None, :]
        s.bundle.est.IO[3:, :] = False                      # per image: cc and pp only (keeps every image well determined)
    s.bundle.serial = None
    buildserialindices(s)
    return s


@pytest.mark.parametrize('kind', ['image-variant-pp', 'two-cameras', 'image-variant-all'])
def test_general_io_blocks(kind):
    """More than one IO block (SURVEY §8 A5: per-image IO columns of multi_res.m:92-111): residual and Jacobian
    (pattern bit-exact), one damped step against the dense solve, GNA / LMP / LM against the oracle, and the
    posterior covariances - the whole hot path through the general-IO kernels (general_io.cu)."""
    s = _general_io_scene(kind)
    x0 = serialize(s)
    W = buildweightmatrix(s)
    P = dbat_b200.Problem(copy.deepcopy(s))
    r = P(x0)
    ro, Jo = brown_euler_cam4(x0, s, True)
    assert relmax(r, ro) < RES_RTOL
    J = P.jacobian(True)
    Jw = Jo.multiply(np.sqrt(W)[:, None]).tocsc()
    Jw.sort_indices()
    assert np.array_equal(J.indptr, Jw.indptr) and np.array_equal(J.indices, Jw.indices)
    np.testing.assert_allclose(J.data, Jw.data, rtol=1e-11, atol=1e-13 * np.abs(Jw.data).max())
    rw = ro * np.sqrt(W)
    N = (Jw.T @ Jw).toarray()
    for lam, jacobi in ((0.0, False), (1e3, False), (0.0, True)):
        p, st = P.normal_step(x0, lam, jacobi)
        po = np.linalg.solve(N + lam * np.eye(N.shape[0]), -(Jw.T @ rw))
        assert relmax(p, po) < 5e-9, (lam, jacobi)
        jp = Jw @ po
        assert abs(st['jp2'] - jp @ jp) <= 1e-9 * (jp @ jp)
        assert abs(st['rjp'] - rw @ jp) <= 1e-9 * abs(rw @ jp)
    P.close()
    for damping in ('gna', 'lmp', 'lm'):
        s1, s2 = copy.deepcopy(s), copy.deepcopy(s)
        s1, ok, it, s0, E = dbat_b200.bundle(s1, damping)
        s2, oko, ito, s0o, Eo = obundle(s2, damping)
        assert ok and oko and E.code == Eo.code == 0
        np.testing.assert_allclose(s0, s0o, rtol=EST_RTOL)
        if damping != 'lm':
            assert it == ito
            np.testing.assert_allclose(E.x, Eo.x, rtol=EST_RTOL, atol=EST_ATOL)
            np.testing.assert_allclose(s1.IO.val, s2.IO.val, rtol=EST_RTOL, atol=EST_ATOL)
        else:
            np.testing.assert_allclose(E.x, Eo.x, rtol=1e-6, atol=1e-9)
        if damping == 'gna':
            for w in ('CIO', 'CEO', 'COP'):
                Cg, Co = dense(dbat_b200.bundle_cov(s1, E, w)), dense(ocov(s2, Eo, w))
                assert Cg.shape == Co.shape and relmax(Cg, Co) < 1e-7, w


def test_full_size_properties():
    """BASELINE config 4 (1000 x 200k x 2M): size-independent properties of one LM pass."""
    s, truth = make_scene(1000, 200000, rays=10)
    P = dbat_b200.Problem(s)
    x0 = dbat_b200.serialize(s)
    p, st = P.normal_step(x0, 0.0, False, trial=True)
    # Gauss-Newton step: J'(Jp+r)=0  =>  r'Jp = -|Jp|^2 ; and the step must reduce f
    assert abs(st['rjp'] + st['jp2']) <= 1e-8 * st['jp2']
    assert st['f_new'] < st['f']
    # predicted decrease of the linear model matches to first order
    assert st['f'] - st['f_new'] > 0.5 * 0.5 * st['jp2']
    # a second evaluation is bit-identical (deterministic assembly)
    p2, st2 = P.normal_step(x0, 1e3, False)
    p3, st3 = P.normal_step(x0, 1e3, False)
    assert st2['f'] == st3['f'] == st['f']
    # residual at the truth is pure measurement noise: sigma0 ~ 1
    s_t = copy.deepcopy(s)
    s_t.IO.val[:] = truth['IO'][:, None]
    s_t.EO.val[:] = truth['EO']
    s_t.OP.val[:] = truth['OP']
    r = P(dbat_b200.serialize(s_t), weighted=True)
    s0 = np.sqrt(r @ r / len(r))
    assert 0.97 < s0 < 1.03
    P.close()


@pytest.mark.parametrize('case', ['model3', 'priors+fixed'])
def test_covariance_statistics_on_the_device(case):
    """dbat_cov_stats (SURVEY §8f N2): posterior standard deviations of every unknown and the pairs of every IO / EO /
    OP block whose correlation exceeds a threshold, computed on the device - against the same statistics taken on
    the host from the oracle's bundle_cov blocks (corrmat.m, high_{eo,op}_correlations.m in block form)."""
    from dbat_b200.report import corrmat
    s, _ = scene(**CASES[case])
    so = copy.deepcopy(s)
    s, ok, it, s0, E = dbat_b200.bundle(s, 'gna')
    so, oko, ito, s0o, Eo = obundle(so, 'gna')
    assert ok and oko
    thres = 0.3                                              # low enough that every kind has pairs
    st = E.problem.cov_stats(s0, thres)
    assert not st['failed']
    ser = s.bundle.serial
    for which, k, key, src, dst in (('CIO', s.IO.val.shape[0], 'io', ser.IO.src, ser.IO.dest),
                                    ('CEO', 6, 'eo', ser.EO.src, ser.EO.dest), ('COP', 3, 'op', ser.OP.src, ser.OP.dest)):
        Co = dense(ocov(so, Eo, which))
        N = Co.shape[0] // k
        B = np.stack([Co[i * k:(i + 1) * k, i * k:(i + 1) * k] for i in range(N)])
        R, sd = corrmat(B, True)
        # standard deviations: element `src` of the stacked parameter array is unknown `dest` of x
        np.testing.assert_allclose(st['std'][np.asarray(dst)], sd.reshape(-1)[np.asarray(src)], rtol=1e-6)
        M = np.tril(np.abs(R), -1) > thres
        n_, c_, r_ = np.nonzero(M.transpose(0, 2, 1))        # block, then column, then row
        r, c, b, v = st[key]
        # the device lists every image's IO block; the oracle's CIO block of an image that shares its camera with an
        # earlier one is the same block: compare all of them
        margin = np.abs(np.abs(R[n_, r_, c_]) - thres) > 1e-6
        assert len(r) == len(r_) or not margin.all()
        if margin.all():
            assert np.array_equal(b, n_) and np.array_equal(r, r_) and np.array_equal(c, c_)
            np.testing.assert_allclose(v, R[n_, r_, c_], rtol=1e-6, atol=1e-9)
    E.problem.close()


def test_full_size_step_against_the_oracle():
    """BASELINE config 4 itself (1000 cameras x 200 000 points x 2 000 000 observations, n = 606 002): one damped
    step of the device against the oracle's sparse solve of the FULL normal equations (J'J + lambda I) p = -J'r as
    the reference forms them (levenberg_marquardt.m:76-82,119) - 1994 Schur clusters, 100 tile columns of the reduced
    system, 36 elimination levels.  Also the residual vector itself (1e-12) and |Jp|^2, r'Jp."""
    import scipy.sparse as sp
    from oracle import lsa
    s, _ = make_scene(1000, 200000, rays=10)
    x0 = serialize(s)
    R = np.sqrt(buildweightmatrix(s))
    P = dbat_b200.Problem(copy.deepcopy(s))
    ro, Jo = brown_euler_cam4(x0, s, True)
    r_dev = P(x0, weighted=False)
    assert np.abs(r_dev - ro).max() <= RES_RTOL * np.abs(ro).max()
    Jw = (sp.diags(R) @ Jo).tocsc()
    rw = R * ro
    N = (Jw.T @ Jw).tocsc()
    n = len(x0)
    nC = n - len(s.bundle.serial.OP.dest)
    lam = 1e-10 * N.diagonal().sum() / n                       # lambda0 of levenberg_marquardt.m:88-106
    po = lsa.solve_spd_pointfirst(N + lam * sp.identity(n, format='csc'), -(Jw.T @ rw), nC)
    p, st = P.normal_step(x0, lam, False)
    assert relmax(p, po) < 5e-9
    jp = Jw @ po
    assert abs(st['f'] - 0.5 * rw @ rw) <= 1e-12 * 0.5 * rw @ rw
    assert abs(st['jp2'] - jp @ jp) <= 1e-9 * (jp @ jp)
    assert abs(st['rjp'] - rw @ jp) <= 1e-9 * abs(rw @ jp)
    p2, _ = P.normal_step(x0, lam, False)
    assert np.array_equal(p, p2), 'default path not bit-reproducible'
    P.close()


@pytest.mark.parametrize('n', [100, 129, 700])
def test_dense_cholesky_solver(n):
    """The reduced-system solver on its own: blocked DMMA Cholesky, folded forward
    substitution, backward solve and explicit inverse against LAPACK."""
    from dbat_b200 import _lib
    rng = np.random.default_rng(n)
    M = rng.standard_normal((n, n + 8))
    A = M @ M.T + 0.5 * n * np.eye(n)
    b = rng.standard_normal(n)
    x, Ai, _ = _lib.dense_chol_solve(A, b, want_inverse=True)
    np.testing.assert_allclose(x, np.linalg.solve(A, b), rtol=1e-10, atol=1e-13)
    Ar = np.linalg.inv(A)
    assert relmax(Ai, Ar) < 1e-10
    with pytest.raises(_lib.DbatError):
        _lib.dense_chol_solve(A - 2 * n * np.eye(n), b)        # not positive definite


def _banded_arrow_spd(n, bw, border, rng, blocks=None):
    """SPD test matrix with the structure of a reduced camera system: a band (or the given list of coupled
    6-column block pairs), `border` dense rows at the end, diagonally dominant."""
    A = np.zeros((n, n))
    if blocks is None:
        for c in range(n):
            lo = max(0, c - bw)
            A[c, lo:c] = rng.standard_normal(c - lo)
    else:
        for a, b in blocks:
            ra, rb = slice(6 * a, min(n, 6 * a + 6)), slice(6 * b, min(n, 6 * b + 6))
            A[ra, rb] = rng.standard_normal((ra.stop - ra.start, rb.stop - rb.start))
        A = np.tril(A, -1)
    if border:
        A[n - border:, :] = rng.standard_normal((border, n))
    A = np.tril(A, -1)
    A = A + A.T
    A += np.diag(np.abs(A).sum(axis=1) + 1.0 + rng.uniform(0, 1, n))
    return A


@pytest.mark.parametrize('n,bw,border,mode', [(50, 50, 0, 0), (423, 423, 0, -1), (700, 90, 9, 0), (2500, 200, 9, 1),
                                              (2500, 200, 9, 2), (6002, 600, 9, 2)])
def test_tile_cholesky_solver(n, bw, border, mode):
    """The sparse tile Cholesky on its own (ordering + symbolic analysis + persistent data-flow kernel +
    backward substitution) against LAPACK on matrices shaped like reduced camera systems."""
    from dbat_b200 import _lib
    rng = np.random.default_rng(n + mode)
    A = _banded_arrow_spd(n, bw, border, rng)
    b = rng.standard_normal(n)
    x, st = _lib.tile_chol_solve(A, b, mode=mode, leaf=40)
    assert st['rc'] == 0
    ref = np.linalg.solve(A, b)
    np.testing.assert_allclose(x, ref, rtol=1e-10, atol=1e-13 * np.abs(ref).max())
    piv = np.diag(np.linalg.cholesky(A))
    assert st['min_pivot'] <= piv.max() and st['max_pivot'] >= piv.min()      # bounds of the true pivots (ordering differs)
    x2, st2 = _lib.tile_chol_solve(A, b, mode=mode, leaf=40, repeat=3)         # epochs: the flags are reused
    np.testing.assert_array_equal(x2, x)
    _, st3 = _lib.tile_chol_solve(A - 2 * np.diag(np.diag(A)), b, mode=mode)
    assert st3['rc'] == _lib.E_NOTSPD


def test_tile_cholesky_dissected_grid():
    """Co-visibility of a 2-D block of images (every image coupled to its neighbours within two grid steps):
    nested dissection gives independent subtrees; the factorisation must not care about the order."""
    from dbat_b200 import _lib
    g = 24
    idx = np.arange(g * g).reshape(g, g)
    blocks = [(int(idx[i, j]), int(idx[k, l])) for i in range(g) for j in range(g)
              for k in range(max(0, i - 2), min(g, i + 3)) for l in range(max(0, j - 2), min(g, j + 3)) if idx[k, l] < idx[i, j]]
    n = 6 * g * g
    rng = np.random.default_rng(4)
    A = _banded_arrow_spd(n, 0, 0, rng, blocks=blocks)
    b = rng.standard_normal(n)
    ref = np.linalg.solve(A, b)
    depth = {}
    for mode in (0, 1, 2):
        x, st = _lib.tile_chol_solve(A, b, mode=mode, leaf=40)
        np.testing.assert_allclose(x, ref, rtol=1e-10, atol=1e-13 * np.abs(ref).max())
        depth[mode] = st['depth']
    assert depth[2] < depth[1]


@pytest.mark.parametrize('model,sigma0', [(-1, 1.62168), (1, 1.68901), (2, 1.68901), (3, 1.6148),
                                          (4, 1.61247), (5, 1.6148)])
def test_camcal_all_models_golden_sigma0(model, sigma0):
    """data/dbat/dbatexports/camcal-dbatreport-model*.txt: sigma0 of the six distortion models
    (camcaldemo_allmodels.m), CUDA path against the reference's golden numbers."""
    s = camcal_struct('default', seed=1)
    s.IO.model.distModel[:] = model
    if abs(model) < 3:
        s.bundle.est.IO[3:5, :] = False
    s, ok, iters, s0, E = dbat_b200.bundle(s, 'gna')
    assert ok
    assert abs(s0 - sigma0) < 6e-6 * (10 if sigma0 == 1.6148 else 1)
    assert E.numParams == (422 if abs(model) < 3 else 423)


@pytest.mark.parametrize('mode', ['maxm'])
def test_schur_fallback_paths_subprocess(mode):
    """The window Schur kernel hands points with more than 20 rays to the per-point kernel.  No small
    scene has such points, so the threshold is lowered (DBAT_GRP_MAXM=6: the 10-ray points of the test
    scene take the per-point kernel, the ragged 3-ray ones stay grouped).  Same step as the oracle."""
    import subprocess
    import sys
    code = r'''
import sys, copy, numpy as np
sys.path.insert(0, %r); sys.path.insert(0, %r)
import dbat_b200
from test_gpu_parity import scene, CASES
from oracle.cameramodel import brown_euler_cam4
from oracle.dbatstruct import buildweightmatrix, serialize
for case in ('priors+fixed', 'ragged'):
    s, _ = scene(**CASES[case])
    x0 = serialize(s); W = buildweightmatrix(s)
    P = dbat_b200.Problem(copy.deepcopy(s))
    p1, st1 = P.normal_step(x0, 10.0, False)
    ro, Jo = brown_euler_cam4(x0, s, True)
    Jw = Jo.multiply(np.sqrt(W)[:, None]).tocsc(); rw = ro * np.sqrt(W)
    N = (Jw.T @ Jw).toarray()
    po = np.linalg.solve(N + 10.0 * np.eye(N.shape[0]), -(Jw.T @ rw))
    assert np.abs(p1 - po).max() / np.abs(po).max() < 5e-9, case
print('FALLBACK-OK')
''' % (os.path.dirname(os.path.dirname(os.path.abspath(__file__))), os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, DBAT_GRP_MAXM='6')
    out = subprocess.run([sys.executable, '-c', code], env=env, capture_output=True, text=True, timeout=600)
    assert 'FALLBACK-OK' in out.stdout, out.stdout + out.stderr


PRAGUE = os.path.join(os.path.dirname(GOLD), 'prague2016cam')
STPIERRE = os.path.join(os.path.dirname(GOLD), 'stpierre')


@pytest.mark.parametrize('stub,sigma0,last', [('weighted', 1.60984, 98.3715), ('fixed', 1.78095, 108.827)])
def test_prague2016_cam_golden_cuda(stub, sigma0, last):
    """BASELINE config 2 data (prague2016 cam, PhotoModeler export, model 1, weighted control points =
    prior OP observations): CUDA path against the reference's golden report and against the oracle."""
    s = loaders.prague_cam_struct(PRAGUE, stub)
    so = copy.deepcopy(s)
    s, ok, iters, s0, E = dbat_b200.bundle(s, 'gna')
    so, oko, iterso, s0o, Eo = obundle(so, 'gna')
    assert ok and oko and iters == iterso
    assert abs(s0 - sigma0) < 6e-6 and abs(E.res[-1] - last) < 6e-4
    np.testing.assert_allclose(E.x, Eo.x, rtol=EST_RTOL, atol=EST_ATOL)
    np.testing.assert_allclose(s0, s0o, rtol=EST_RTOL)
    for w in ('CEO', 'COP'):
        Cg = dbat_b200.bundle_cov(s, E, w).toarray()
        Co = dense(ocov(so, Eo, w))
        assert relmax(Cg, Co) < 1e-8


@pytest.mark.parametrize('damping', ['lmp', 'lm', 'gna'])
def test_prague2016_selfcalibration(damping):
    """BASELINE config 2 as stated: Brown self-calibration on the prague2016 data with LMP damping
    (no reference golden exists for this variant: oracle vs CUDA)."""
    s = loaders.prague_cam_struct(PRAGUE, 'weighted')
    s.IO.model.distModel[:] = 3
    s.bundle.est.IO[:] = True
    s.bundle.est.IO[4, :] = False
    so = copy.deepcopy(s)
    s, ok, iters, s0, E = dbat_b200.bundle(s, damping)
    so, oko, iterso, s0o, Eo = obundle(so, damping)
    assert ok and oko
    np.testing.assert_allclose(s0, s0o, rtol=EST_RTOL)
    if damping != 'lm':
        assert iters == iterso
        np.testing.assert_allclose(E.x, Eo.x, rtol=EST_RTOL, atol=EST_ATOL)
    else:
        np.testing.assert_allclose(E.x, Eo.x, rtol=1e-6, atol=1e-9)


@pytest.mark.parametrize('damping', ['gna', 'lmp', 'lm'])
def test_stpierre_selfcalibration(damping):
    """BASELINE config 3 data (hamburg2017 StPierre, `C5_reduced` PhotoModeler export: 28 images, 2003
    object points, 4331 image points, 4 weighted control points) set up like `stpierrebundledemo_ps.m`:
    forward Brown model (-1), self-calibration of everything but skew/aspect, datum from the prior
    observations of the control points; followed by bundle_cov.  The reference holds no golden for
    this input (the demo's .psz is missing, the export has no image size): oracle vs CUDA."""
    s = loaders.stpierre_struct(STPIERRE)
    so = copy.deepcopy(s)
    s, ok, iters, s0, E = dbat_b200.bundle(s, damping)
    so, oko, iterso, s0o, Eo = obundle(so, damping)
    assert ok and oko
    np.testing.assert_allclose(s0, s0o, rtol=EST_RTOL)
    assert abs(s0 - 1.0282960127) < 1e-8                   # value of the oracle at the time of writing
    if damping != 'lm':
        assert iters == iterso
        np.testing.assert_allclose(E.x, Eo.x, rtol=EST_RTOL, atol=EST_ATOL)
        np.testing.assert_allclose(E.res, Eo.res, rtol=1e-9)
    else:
        np.testing.assert_allclose(E.x, Eo.x, rtol=1e-6, atol=1e-9)
    if damping == 'gna':
        for w in ('CIO', 'CEO', 'COP'):
            Cg = dbat_b200.bundle_cov(s, E, w).toarray()
            Co = dense(ocov(so, Eo, w))
            assert relmax(Cg, Co) < 1e-7, w
            sg, sd = np.sqrt(np.diag(Cg)), np.sqrt(np.diag(Co))
            m = sd > 0
            np.testing.assert_allclose(sg[m], sd[m], rtol=1e-7)


@pytest.mark.parametrize('seed', [1, 2, 3, 4, 5, 6])
def test_structural_rank_matches_oracle_on_thin_networks(seed):
    """sprank(J)<n (code -4) on thinned networks (some points keep a single ray; on even seeds those
    points are fixed, which restores full structural rank): same verdict as the oracle's
    structural_rank of the same Jacobian."""
    rng = np.random.default_rng(seed)
    s, _ = make_scene(8, 60, rays=3, seed=20 + seed, build_indices=False)
    keep = rng.random(len(s.IP.img)) < 0.9
    for f in ('val', 'std'):
        setattr(s.IP, f, getattr(s.IP, f)[:, keep])
    for f in ('img', 'op', 'cam'):
        setattr(s.IP, f, getattr(s.IP, f)[keep])
    cnt = np.bincount(s.IP.op, minlength=s.OP.val.shape[1])
    if seed % 2 == 0:
        s.bundle.est.OP[:, cnt < 2] = False
    s.bundle.est.OP[:, cnt == 0] = False
    buildserialindices(s)
    so = copy.deepcopy(s)
    s, ok, _, _, E = dbat_b200.bundle(s, 'gna')
    so, oko, _, _, Eo = obundle(so, 'gna')
    assert (E.code == -4) == (Eo.code == -4), (E.code, Eo.code)
    assert E.code == Eo.code


# ------------------------------------------------------------------ start values (SURVEY §8f N1)
def test_forwintersect_matches_oracle_camcal():
    """forwintersect(s,'all',true) as in camcaldemo.m:107 on the camcal project (golden EO, calibrated
    camera): CUDA kernel vs the literal restatement of pm_multiforwintersect / pm_forwintersect3."""
    from oracle.photogrammetry import forwintersect as ofwi
    from camcal_fixture import camcal_struct
    s = camcal_struct('golden', 0)
    s.OP.val[:, s.bundle.est.OP.all(axis=0)] = np.nan          # unknown before the intersection
    sg, idg, resg = dbat_b200.forwintersect(s, 'all', True)
    so, ido, reso = ofwi(s, 'all', True)
    assert np.array_equal(idg, ido) and len(idg) == 96
    est = s.bundle.est.OP.all(axis=0)
    np.testing.assert_allclose(sg.OP.val[:, est], so.OP.val[:, est], rtol=1e-9, atol=1e-9)
    np.testing.assert_allclose(resg, reso, rtol=1e-6, atol=1e-10)
    assert np.array_equal(sg.OP.val[:, ~est], s.OP.val[:, ~est])       # control points untouched


@pytest.mark.parametrize('case', ['model3', 'ragged'])
def test_forwintersect_matches_oracle_synthetic(case):
    """Same on seeded synthetic blocks (ragged: points with different ray counts, incl. an explicit id list
    and a point left with a single ray -> NaN)."""
    from oracle.photogrammetry import forwintersect as ofwi
    s, truth = scene(**CASES[case])
    s.IO.val[5:10, :] = truth['IO'][5:10, None]                 # non-trivial lens correction
    k = np.flatnonzero(s.IP.op == 3)
    keep = np.ones(len(s.IP.op), bool)
    keep[k[1:]] = False                                          # point 3 keeps one ray
    for f in ('val', 'std'):
        setattr(s.IP, f, getattr(s.IP, f)[:, keep])
    for f in ('img', 'op', 'cam'):
        setattr(s.IP, f, getattr(s.IP, f)[keep])
    ids = np.arange(0, s.OP.val.shape[1], 2)
    ids = np.union1d(ids, [3])
    sg, idg, resg = dbat_b200.forwintersect(s, ids)
    so, ido, reso = ofwi(s, ids)
    assert np.array_equal(idg, ido)
    assert np.isnan(sg.OP.val[:, 3]).all() and np.isnan(so.OP.val[:, 3]).all()
    m = ~np.isnan(so.OP.val[0])
    np.testing.assert_allclose(sg.OP.val[:, m], so.OP.val[:, m], rtol=1e-9, atol=1e-9)
    mr = ~np.isnan(reso)
    np.testing.assert_allclose(resg[mr], reso[mr], rtol=1e-6, atol=1e-10)
    assert np.isnan(resg[~mr]).all()


def test_forwintersect_refuses_bad_eo():
    s, _ = scene(**CASES['model3'])
    s.EO.val[0, 0] = np.nan
    with pytest.raises(ValueError, match='EO'):
        dbat_b200.forwintersect(s, 'all')


def test_resect_matches_oracle_camcal():
    """resect(s0,'all',cpId,1,0,cpId) as in camcaldemo.m:102 / parseops.m:38 on the camcal script project
    (default camera, EO unknown): batched 3-point resection kernel vs the restatement of resect.m /
    pm_resect_3pt.m."""
    from oracle.photogrammetry import resect as oresect
    s = loaders.load_camcal_script(os.path.join(os.path.dirname(GOLD), 'camcaldemo'))
    cpId = np.asarray(s.OP.id)[s.prior.OP.isCtrl]
    sg, rmsg, failg = dbat_b200.resect(s, 'all', cpId, 1, 0, cpId)
    so, rmso, failo = oresect(s, 'all', cpId, 1, 0, cpId)
    assert not failg and not failo
    np.testing.assert_allclose(sg.EO.val, so.EO.val, rtol=1e-7, atol=1e-8)
    np.testing.assert_allclose(rmsg, rmso, rtol=1e-6, atol=1e-12)
    # two candidate triangles per camera (n = 2): same winner
    sg2, rmsg2, _ = dbat_b200.resect(s, [0, 5, 20], cpId, 2, 0.5, cpId)
    so2, rmso2, _ = oresect(s, [0, 5, 20], cpId, 2, 0.5, cpId)
    np.testing.assert_allclose(sg2.EO.val[:, [0, 5, 20]], so2.EO.val[:, [0, 5, 20]], rtol=1e-7, atol=1e-8)
    np.testing.assert_allclose(rmsg2, rmso2, rtol=1e-6, atol=1e-12)


def test_camcal_script_pipeline_on_device_matches_golden_report():
    """The camcal script's operations on the device - spatial_resection, forward_intersection,
    bundle_adjustment - against the reference's report.txt: 8 iterations, first error 28805.9, last error
    98.556, sigma0 1.6148 (the first error depends on the start values only)."""
    s = loaders.load_camcal_script(os.path.join(os.path.dirname(GOLD), 'camcaldemo'))
    cpId = np.asarray(s.OP.id)[s.prior.OP.isCtrl]
    s1, rms, fail = dbat_b200.resect(s, 'all', cpId, 1, 0, cpId)
    assert not fail
    s2, ids, res = dbat_b200.forwintersect(s1, 'all', True)
    assert np.isfinite(s2.OP.val).all()
    s3, ok, iters, sigma0, E = dbat_b200.bundle(s2, 'gna')
    assert ok and iters == 8
    assert abs(E.res[0] - 28805.9) < 0.06 and abs(E.res[-1] - 98.556) < 6e-4
    assert abs(sigma0 - 1.6148) < 6e-5


def test_resect_reports_failure_with_two_control_points():
    s = loaders.load_camcal_script(os.path.join(os.path.dirname(GOLD), 'camcaldemo'))
    cpId = np.asarray(s.OP.id)[s.prior.OP.isCtrl][:2]
    sg, rms, fail = dbat_b200.resect(s, [0, 1], cpId, 1, 0, cpId)
    assert fail and np.isnan(sg.EO.val[:, [0, 1]]).all() and np.isinf(rms).all()


@pytest.mark.parametrize('case', ['model3', 'priors+fixed', 'ragged'])
def test_gauss_markov_direct_call(case):
    """gauss_markov.m called directly (numeric convTol; via bundle() the reference passes a function
    handle and fails): same iterates, iteration count and residual norms as the restatement."""
    from oracle.lsa import gauss_markov as ogm
    s, _ = scene(**CASES[case])
    x0 = serialize(s)
    W = buildweightmatrix(s)
    P = dbat_b200.Problem(copy.deepcopy(s))
    # sTest off: on the unscaled J'J of a self-calibrating bundle MATLAB's rcond warning fires (and the
    # restatement's emulation with it), which is exactly why the other optimisers scale the columns
    x, code, n, final, T, rr = dbat_b200.gauss_markov(P, x0, W, 20, 1e-6, False, False)
    xo, codeo, no, finalo, To, rro = ogm(lambda xx, j: brown_euler_cam4(xx, s, j), x0, W, 20, 1e-6, False, False)
    assert code == codeo == 0 and n == no
    np.testing.assert_allclose(x, xo, rtol=EST_RTOL, atol=EST_ATOL)
    np.testing.assert_allclose(rr, rro, rtol=1e-10)
    np.testing.assert_allclose(T, To, rtol=1e-8, atol=1e-10)
    np.testing.assert_allclose(final.weighted.r, finalo.weighted.r, rtol=1e-9, atol=1e-11)
    P.close()


CAMCALPM = os.path.join(os.path.dirname(GOLD), 'camcalpm')


@pytest.mark.parametrize('pm,iters,first,last,sigma0,nparams', [
    ('camcal-pmexport.txt', 9, 30873.9, 98.556, 1.6148, 423),
    ('camcal-pmexport5.txt', 6, 254.75, 18.4099, 2.80749, 57)])
def test_camcal_pm_demo_pipeline_on_device(pm, iters, first, last, sigma0, nparams):
    """camcaldemo.m / camcaldemo2.m end to end on the device (resect, forwintersect, bundle GNA) against
    the reference's reports: iteration count, last error, sigma0, number of parameters to the printed
    digits; the first error (a function of the start values only) to 1e-5: the Grunert quartic of image 21
    has a nearly double root, where the device's polynomial solver and MATLAB's eigenvalue-based `roots`
    (which the restatement reproduces: 30873.87) differ by 4e-6 in the resected pose."""
    s = loaders.camcal_pm_struct(os.path.join(CAMCALPM, pm), os.path.join(CAMCALPM, 'camcal-fixed.txt'))
    cpId = np.asarray(s.OP.id)[s.prior.OP.isCtrl]
    s1, _, fail = dbat_b200.resect(s, 'all', cpId, 1, 0, cpId)
    assert not fail
    s2, _, _ = dbat_b200.forwintersect(s1, 'all', True)
    s3, ok, it, s0, E = dbat_b200.bundle(s2, 'gna')
    assert ok and it == iters and E.numParams == nparams
    assert abs(E.res[0] - first) < 1e-5 * first
    assert abs(E.res[-1] - last) < 0.6 * 10 ** (np.floor(np.log10(last)) - 5)
    assert abs(s0 - sigma0) < 0.6 * 10 ** (np.floor(np.log10(sigma0)) - 5)


def test_camcal_missing_obs_demo_on_device():
    """camcaldemo_missing_obs.m on the device: failure code -4 at iteration 0, first error 30118.6,
    sigma0 499.142 as in the reference's report."""
    s = loaders.camcal_pm_struct(os.path.join(CAMCALPM, 'camcal-pmexport-missing-obs.txt'),
                                 os.path.join(CAMCALPM, 'camcal-fixed.txt'))
    cpId = np.asarray(s.OP.id)[s.prior.OP.isCtrl]
    s1, _, fail = dbat_b200.resect(s, 'all', cpId, 1, 0, cpId)
    s2, _, _ = dbat_b200.forwintersect(s1, 'all', True)
    s3, ok, it, s0, E = dbat_b200.bundle(s2, 'gna')
    assert not ok and it == 0 and E.code == -4 and E.numParams == 423
    assert abs(E.res[0] - 30118.6) < 1e-5 * 30118.6 and abs(s0 - 499.142) < 1e-5 * 499.142
