"""Posterior covariances (dbat_cov, dbat_cov_stats) at the sizes real projects reach, and the dense inverse they use.

The covariance stack is separate from the step: the undamped, Jacobi-scaled reduced system is copied out of the tiles
(k_tc_to_dense), factored and inverted densely (chol_factor + chol_inverse), and the inverse is consumed by k_cop /
k_cop_gen (COP), k_cov_rows / k_cov_U / k_cov_pp (CXX, COPF) or k_cam_blocks + k_block_corr (cov_stats).

Every case compares at a fixed x (the start values) with s0 = 1, so that no optimiser run enters: the device's
covariances of P(x0) against oracle.bundle.bundle_cov on the oracle's weighted Jacobian at the same x0.  Elements are
compared scale-free, |dC_ab| <= TOL sqrt(C_aa C_bb), standard deviations at rtol STD_RTOL.
"""
import copy
from types import SimpleNamespace as NS

import numpy as np
import pytest
import scipy.linalg as sla
import scipy.sparse as sp

pytestmark = pytest.mark.gpu

import dbat_b200
from dbat_b200 import _lib as dlib
from dbat_b200.report import corrmat
from dbat_b200.synth import make_scene
from oracle.bundle import BLOCK_PATH_ABOVE, bundle_cov as ocov
from oracle.cameramodel import brown_euler_cam4
from oracle.dbatstruct import buildserialindices, buildweightmatrix, serialize

TOL = 1e-8
STD_RTOL = 1e-9
EPS = np.finfo(float).eps


@pytest.fixture(scope='module', autouse=True)
def _lib(built_lib):
    return built_lib


# --------------------------------------------------------------------------------------------- helpers
def oracle_e(s, x0):
    """The fields of the oracle's bundle result that bundle_cov reads, at x0 with s0 = 1."""
    _, J = brown_euler_cam4(x0, s, True)
    Jw = (sp.diags(np.sqrt(buildweightmatrix(s))) @ J).tocsc()
    return NS(x=x0, s0=1.0, final=NS(weighted=NS(J=Jw), factorized=None))


def diag_blocks(M, k):
    """(N, k, k) diagonal blocks of a (k N)^2 matrix, dense or sparse."""
    N = M.shape[0] // k
    if sp.issparse(M):
        M = M.tocoo()
        m = M.row // k == M.col // k
        B = np.zeros((N, k, k))
        B[M.row[m] // k, M.row[m] % k, M.col[m] % k] = M.data[m]
        return B
    M = np.asarray(M).reshape(N, k, N, k)
    i = np.arange(N)
    return M[i, :, i, :]


def cam_blocks(s, F, key):
    """CIO / CEO diagonal blocks straight from the block factor's Cc (what _cov_blocks spreads into a full matrix)."""
    des = getattr(s.bundle.deserial, key)
    k, N = getattr(s.bundle.est, key).shape
    pos = np.full(int(max(F.camx.max(), F.opx.max())) + 1, -1)
    pos[F.camx] = np.arange(len(F.camx))
    cm = np.full(k * N, -1)
    cm[des.dest] = pos[des.src]
    cm = cm.reshape(N, k)
    ok = (cm[:, :, None] >= 0) & (cm[:, None, :] >= 0)
    return np.where(ok, F.Cc[np.maximum(cm, 0)[:, :, None], np.maximum(cm, 0)[:, None, :]], 0.0)


def cop_from_factor(F, pts):
    """COP of the listed points, point by point from the block factor: Ai_j + Y_j' Cc Y_j."""
    order = np.argsort(F.pt, kind='stable')
    start = np.searchsorted(F.pt[order], np.arange(int(F.pt.max()) + 2))
    Y = F.Y.tocsc()
    out = np.zeros((len(pts), 3, 3))
    for q, j in enumerate(pts):
        cols = order[start[j]:start[j + 1]]
        if len(cols) == 0:
            continue
        Yj = Y[:, cols].tocoo()
        rows, ri = np.unique(Yj.row, return_inverse=True)
        Yd = np.zeros((len(rows), len(cols)))
        Yd[ri, Yj.col] = Yj.data
        c = F.comp[cols]
        out[q][np.ix_(c, c)] = F.Ai[j][np.ix_(c, c)] + Yd.T @ F.Cc[np.ix_(rows, rows)] @ Yd
    return out


def assert_cov(Cg, Co, what, tol=TOL):
    """|Cg - Co| <= tol sqrt(Co_aa Co_bb) elementwise over the last two axes; zero rows / columns stay exactly zero."""
    Cg, Co = np.asarray(Cg), np.asarray(Co)
    assert Cg.shape == Co.shape, (what, Cg.shape, Co.shape)
    d = np.sqrt(np.abs(np.diagonal(Co, axis1=-2, axis2=-1)))
    scale = d[..., :, None] * d[..., None, :]
    err = np.abs(Cg - Co)
    assert np.all(np.isfinite(Cg)), what
    assert np.all(err[scale == 0] == 0), what
    rel = err[scale > 0] / scale[scale > 0]
    assert rel.size == 0 or rel.max() <= tol, '%s: max scale-free error %.3g' % (what, rel.max())
    sg = np.sqrt(np.diagonal(Cg, axis1=-2, axis2=-1))
    np.testing.assert_allclose(sg[d > 0], d[d > 0], rtol=STD_RTOL, err_msg=what)


def std_from_blocks(s, blocks):
    """Standard deviation of every unknown (x order) from the IO / EO / OP diagonal blocks."""
    ser = s.bundle.serial
    std = np.full(len(serialize(s)), np.nan)
    for key, B in blocks.items():
        sd = np.sqrt(np.diagonal(B, axis1=1, axis2=2)).reshape(-1)
        sr = getattr(ser, key)
        std[np.asarray(sr.dest)] = sd[np.asarray(sr.src)]
    return std


def pick_threshold(Rs):
    """A correlation threshold in [0.3, 0.9] that no correlation of the blocks comes within 1e-6 of."""
    v = np.concatenate([np.abs(R[:, np.tril_indices(R.shape[1], -1)[0], np.tril_indices(R.shape[1], -1)[1]]).ravel()
                        for R in Rs])
    v = np.sort(v[np.isfinite(v)])                    # rows of fixed elements have no correlation
    for t in np.linspace(0.3, 0.9, 601):
        i = np.searchsorted(v, t)
        near = [abs(v[j] - t) for j in (i - 1, i) if 0 <= j < len(v)]
        if min(near) > 1e-6:
            return float(t)
    raise AssertionError('no threshold with a margin')


def check_cov_stats(P, s, blocks, with_lists=True):
    """cov_stats(1, thres): std of every unknown, and the IO / EO / OP hit lists as corrmat + high_*_correlations
    form them from the oracle's blocks (block, then column, then row)."""
    Rs = {k: corrmat(B, True)[0] for k, B in blocks.items()}
    thres = pick_threshold(list(Rs.values())) if with_lists else 0.95
    st = P.cov_stats(1.0, thres)
    assert not st['failed']
    ref = std_from_blocks(s, blocks)
    np.testing.assert_allclose(st['std'], ref, rtol=STD_RTOL)
    if not with_lists:
        return
    for key, R in Rs.items():
        M = np.tril(np.abs(R), -1) > thres
        n_, c_, r_ = np.nonzero(M.transpose(0, 2, 1))
        r, c, b, v = st[key.lower()]
        assert np.array_equal(b, n_) and np.array_equal(r, r_) and np.array_equal(c, c_), key
        np.testing.assert_allclose(v, R[n_, r_, c_], rtol=1e-6, atol=1e-9)


def elimination_order(s):
    """Images in the order the device's reduced system holds them (the host symbolic analysis dbat_create runs)."""
    nImg, nOP = s.EO.val.shape[1], s.OP.val.shape[1]
    nEO = s.bundle.est.EO[:6].sum(axis=0).astype(np.int64)
    sym = dlib.tile_symbolic(s.IP.img, s.IP.op, nImg, nOP, nEO, len(s.bundle.serial.IO.dest), xyz=s.EO.val[0:3])
    has = nEO > 0
    return np.flatnonzero(has)[np.argsort(sym['imgS'][has], kind='stable')], sym


# --------------------------------------------------------------------------------------------- the dense inverse
def _spd(n, family, rng):
    """(A, cond): M M' + c I (well conditioned), or a unit-diagonal matrix of condition about 1e8 (what the
    Jacobi-scaled reduced system looks like)."""
    if family == 'mmt':
        M = rng.standard_normal((n, n + 8))
        A = M @ M.T + 0.5 * n * np.eye(n)
    else:
        Q = np.linalg.qr(rng.standard_normal((n, n)))[0] if n > 1 else np.ones((1, 1))
        A = (Q * np.logspace(0, -8, n)) @ Q.T
        d = 1.0 / np.sqrt(np.diag(A))
        A = A * d[:, None] * d[None, :]
    A = 0.5 * (A + A.T)
    ev = np.linalg.eigvalsh(A)
    return A, ev[-1] / ev[0]


@pytest.mark.parametrize('family', ['mmt', 'unitdiag-1e8'])
@pytest.mark.parametrize('n', [1, 2, 100, 127, 128, 129, 255, 256, 511, 512, 513, 700, 1000, 6001])
def test_dense_chol_inverse(n, family):
    """chol_factor + chol_inverse on their own at every padding situation of the last block (rhs row with no padding
    at n = 127, a full padding block at n = 128, ...), from one block to the size of BASELINE config 4's reduced
    system."""
    rng = np.random.default_rng(1000 + n)
    A, cond = _spd(n, family, rng)
    bound = 64 * np.sqrt(n) * cond * EPS
    Ai, _ = dlib.dense_chol_inverse(A, repeat=1)
    Ar = sla.inv(A)
    err = np.max(np.abs(Ai - Ar)) / np.max(np.abs(Ar))
    assert err <= bound, err / (cond * EPS)
    Ai3, _ = dlib.dense_chol_inverse(A, repeat=3)
    assert np.array_equal(Ai3, Ai)
    # the first pivot not positive
    with pytest.raises(dlib.DbatError):
        dlib.dense_chol_inverse(A - 2 * A[0, 0] * np.eye(n))
    # only the last pivot (index n - 1) not positive
    Ab = A.copy()
    if n == 1:
        Ab[0, 0] = -1.0
    else:
        a = A[:n - 1, n - 1]
        Ab[n - 1, n - 1] = a @ sla.cho_solve(sla.cho_factor(A[:n - 1, :n - 1], lower=True), a) - 1e-3 * A[n - 1, n - 1]
    with pytest.raises(dlib.DbatError):
        dlib.dense_chol_inverse(Ab)


# --------------------------------------------------------------------------------------------- block-path scenes
def _general_io(s, kind):
    nImg = s.IO.val.shape[1]
    if kind == 'image-variant-pp':
        s.IO.struct.block[1:3, :] = np.arange(1, nImg + 1)
    elif kind == 'two-cameras':
        cam = (np.arange(nImg) % 2) + 1
        s.IO.struct.block[:] = cam[None, :]
        s.IO.val[0, cam == 2] *= 1.01
        s.IO.val[1, cam == 2] += 0.05
    s.bundle.serial = None
    buildserialindices(s)
    return s


BLOCK_SCENES = {
    'mid': dict(nImg=100, nOP=20000, seed=20240607),
    'wide': dict(nImg=400, nOP=40000),
    'gio-two-cameras': dict(nImg=100, nOP=20000, seed=20240607, io='two-cameras'),
    'gio-image-variant-pp': dict(nImg=100, nOP=20000, seed=20240607, io='image-variant-pp'),
}


def _block_scene(name):
    c = dict(BLOCK_SCENES[name])
    io = c.pop('io', None)
    s, _ = make_scene(c.pop('nImg'), c.pop('nOP'), rays=10, **c)
    return _general_io(s, io) if io else s


@pytest.mark.parametrize('name', list(BLOCK_SCENES))
def test_block_path_covariances(name):
    """CIO / CEO / COP and cov_stats of a 1/10-scale and a 400-image project (k_cop over 20 000 and 40 000 points, a
    dissected tiled system copied to dense, chol_inverse over 5 and 19 blocks), and of the general-IO set-ups at
    100 x 20 000 (k_cop_gen, k_cam_blocks with per-image IO columns), against the oracle's block elimination."""
    s = _block_scene(name)
    x0 = serialize(s)
    n = len(x0)
    assert n > BLOCK_PATH_ABOVE
    P = dbat_b200.Problem(copy.deepcopy(s))
    info = P.reduced_info()
    if name == 'wide':
        assert (info['ld'] + 127) // 128 >= 19
    P(x0)
    dev = {k: P.cov(k, 1.0) for k in ('cio', 'ceo', 'cop')}
    e = oracle_e(s, x0)
    Cop = diag_blocks(ocov(s, e, 'COP'), 3)
    F = e.final.factorized
    assert F.blocks and not F.fail
    blocks = {'IO': cam_blocks(s, F, 'IO'), 'EO': cam_blocks(s, F, 'EO'), 'OP': Cop}
    assert_cov(dev['cio'], blocks['IO'], 'CIO')
    assert_cov(dev['ceo'], blocks['EO'], 'CEO')
    assert_cov(dev['cop'], Cop, 'COP')
    check_cov_stats(P, s, blocks)
    P.close()


def test_mid_covariance_against_a_direct_solve():
    """The Schur formula itself, not only its implementation: 3 x 3 COP blocks of 20 points of the mid scene from a
    sparse LU solve N X = E_j of the full normal matrix, for the points of the first and the last image of the
    elimination order, the points with the fewest and the most rays, and a seeded sample."""
    import scipy.sparse.linalg as spla
    s = _block_scene('mid')
    x0 = serialize(s)
    order, sym = elimination_order(s)
    rays = np.bincount(s.IP.op, minlength=s.OP.val.shape[1])
    first, last = s.IP.op[s.IP.img == order[0]], s.IP.op[s.IP.img == order[-1]]
    rng = np.random.default_rng(5)
    pts = [first[0], first[-1], last[0], last[-1], int(np.argmin(rays)), int(np.argmax(rays))]
    pts = list(dict.fromkeys(pts))
    pts += list(rng.choice(np.setdiff1d(np.arange(len(rays)), pts), 20 - len(pts), replace=False))
    P = dbat_b200.Problem(copy.deepcopy(s))
    info = P.reduced_info()
    assert (info['ld'], info['nS']) == (sym['ld'], sym['nS'])
    P(x0)
    Cg = P.cov('cop', 1.0)[pts]
    P.close()
    e = oracle_e(s, x0)
    N = (e.final.weighted.J.T @ e.final.weighted.J).tocsc()
    opx = np.zeros((len(rays), 3), np.int64)
    src, dest = np.asarray(s.bundle.serial.OP.src), np.asarray(s.bundle.serial.OP.dest)
    opx[src // 3, src % 3] = dest
    cols = opx[pts].ravel()
    E = np.zeros((N.shape[0], len(cols)))
    E[cols, np.arange(len(cols))] = 1.0
    # solved Jacobi-scaled: on the unscaled N, SuperLU's own error reaches 1.4e-9 in the standard deviations, scaled it
    # agrees with the oracle's block elimination to 1.4e-11
    D = 1.0 / np.sqrt(N.diagonal())
    X = D[:, None] * spla.splu((sp.diags(D) @ N @ sp.diags(D)).tocsc()).solve(D[:, None] * E)
    Cd = np.stack([X[cols[3 * q:3 * q + 3], 3 * q:3 * q + 3] for q in range(len(pts))])
    assert_cov(Cg, 0.5 * (Cd + Cd.transpose(0, 2, 1)), 'COP vs direct solve')


# --------------------------------------------------------------------------------------------- dense-oracle scenes
def _edge_scene(nImg, nIO):
    """make_scene with nIO estimated IO elements: 9 by default, 8 with K3 fixed, 10 with skew estimated."""
    s, _ = make_scene(nImg, 60, rays=8, seed=5, build_indices=False)
    if nIO == 8:
        s.bundle.est.IO[7, :] = False
    elif nIO == 10:
        s.bundle.est.IO[4, :] = True
    buildserialindices(s)
    return s


# (nImg, nIO) -> reduced system: nS real unknowns, tile ld (the rhs row sits at ld - 1), dense copy ldd = ld rounded
# up to 128
EDGES = {
    'ld128-rhs-last-row': (21, 8, dict(nS=127, ld=128)),          # ldd = ld, no padding at all: rhs row = last row
    'ld64mod128-rhs-last-row': (10, 10, dict(nS=63, ld=64)),      # nS = ld - 1, then 64 rows of dense padding
    'ld64mod128-tile-padding': (21, 9, dict(nS=128, ld=192)),     # 63 rows of tile padding, 64 of dense padding
    'ld128-tile-padding': (15, 9, dict(nS=92, ld=128)),
}


@pytest.mark.parametrize('edge', list(EDGES))
def test_block_edges_of_the_dense_copy(edge):
    """The padding and rhs-row handling of cov_factor (k_dense_unit_diag, chol_factor at ldd = ld rounded up to 128)
    where the rhs row ld - 1 is the dense matrix's last row, where 64 padding rows follow it, and where no tile padding
    sits between the last unknown and the rhs row: CEO / COP / CXX against the dense oracle."""
    nImg, nIO, want = EDGES[edge]
    s = _edge_scene(nImg, nIO)
    x0 = serialize(s)
    P = dbat_b200.Problem(copy.deepcopy(s))
    info = P.reduced_info()
    assert (info['nS'], info['ld']) == (want['nS'], want['ld'])
    P(x0)
    dev = {k: P.cov(k, 1.0) for k in ('cio', 'ceo', 'cop', 'cxx')}
    P.close()
    e = oracle_e(s, x0)
    for k, w in (('cio', 'CIO'), ('ceo', 'CEO'), ('cop', 'COP')):
        assert_cov(dev[k], diag_blocks(ocov(s, e, w), dev[k].shape[1]), w)
    assert_cov(dev['cxx'], ocov(s, e, 'CXX'), 'CXX')


@pytest.mark.parametrize('nOP', [65535, 66000])
def test_dense_point_covariance_with_many_object_points(nOP):
    """CXX / CXX_OP / COP of a project with more object points than a grid's y dimension holds (65 535), of which
    only the first 1 500 are estimated and the rest are fixed at their true coordinates."""
    s, truth = make_scene(30, nOP, rays=3, seed=31, build_indices=False)
    assert np.bincount(s.IP.op, minlength=nOP).min() >= 2
    s.bundle.est.OP[:, 1500:] = False
    s.OP.val[:, 1500:] = truth['OP'][:, 1500:]
    buildserialindices(s)
    x0 = serialize(s)
    n = len(x0)
    m3 = len(s.bundle.serial.OP.dest)
    assert m3 == 4500 and n <= BLOCK_PATH_ABOVE
    P = dbat_b200.Problem(copy.deepcopy(s))
    P(x0)
    dev = {k: P.cov(k, 1.0) for k in ('cxx', 'cxx_op', 'cop')}
    P.close()
    e = oracle_e(s, x0)
    Cxx = ocov(s, e, 'CXX')
    assert_cov(dev['cxx'], Cxx, 'CXX')
    assert_cov(dev['cxx_op'], Cxx[n - m3:, n - m3:], 'CXX_OP')
    ser = s.bundle.serial.OP
    cop = np.zeros((nOP, 3, 3))
    opx = np.full((nOP, 3), -1)
    opx[np.asarray(ser.src) // 3, np.asarray(ser.src) % 3] = ser.dest
    for j in range(1500):
        c = np.flatnonzero(opx[j] >= 0)
        cop[j][np.ix_(c, c)] = Cxx[np.ix_(opx[j, c], opx[j, c])]
    assert_cov(dev['cop'], cop, 'COP')


# --------------------------------------------------------------------------------------------- BASELINE config 4
def test_config4_covariances():
    """BASELINE config 4 (1000 x 200 000 x 2 000 000): chol_inverse at 47 blocks.  Full CEO / CIO and the
    standard deviations of the camera unknowns against the oracle's block elimination; COP of a seeded sample of
    4 096 points and of every point of two images, point by point from the block factor (the oracle's full COP
    loop is about 4e13 flops on the host)."""
    from oracle.bundle import _prepare_blocks
    s, _ = make_scene(1000, 200000, rays=10)
    x0 = serialize(s)
    P = dbat_b200.Problem(copy.deepcopy(s))
    info = P.reduced_info()
    assert (info['ld'] + 127) // 128 >= 47
    P(x0)
    dev = {k: P.cov(k, 1.0) for k in ('cio', 'ceo', 'cop')}
    st = P.cov_stats(1.0, 0.95)
    P.close()
    assert not st['failed']
    e = oracle_e(s, x0)
    _prepare_blocks(s, e)
    F = e.final.factorized
    assert not F.fail
    assert_cov(dev['cio'], cam_blocks(s, F, 'IO'), 'CIO')
    assert_cov(dev['ceo'], cam_blocks(s, F, 'EO'), 'CEO')
    np.testing.assert_allclose(st['std'][F.camx], np.sqrt(np.diag(F.Cc)), rtol=STD_RTOL)
    rng = np.random.default_rng(47)
    nOP = s.OP.val.shape[1]
    pts = np.unique(np.concatenate([rng.choice(nOP, 4096, replace=False), s.IP.op[s.IP.img == 0],
                                    s.IP.op[s.IP.img == 999]]))
    assert_cov(dev['cop'][pts], cop_from_factor(F, pts), 'COP')
