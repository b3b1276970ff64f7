"""The sparse tile Cholesky on the device (csrc/tilechol.cu: k_tchol_factor with tc_potrf64 / tc_diag16, then
k_tchol_bwd) against a plain LAPACK reference of the same operation.

dbat_tile_chol_solve runs the ordering, the symbolic analysis and the data-flow kernels on a caller-given SPD
matrix whose 6-column blocks play the images.  Its elimination order is recovered without a device: the same
co-visibility graph (one two-image point per coupled pair of blocks) goes through dbat_tile_symbolic, whose counts
must agree with the solver's, and imgS then gives the permutation P.  The criteria:
- backward error eta = ||b - A x||_inf / (||A||_inf ||x||_inf + ||b||_inf), residual in long double, within
  ETA_FACTOR of LAPACK's on the same system: independent of the conditioning, so it holds for every family;
- forward error against LAPACK at 1e-12 and the exact pivot statistics (min / max of diag(chol(P A P')) over the
  real unknowns, neither the padding's 1 nor the rhs row's ~1e150) where cond(A) <= 1e4;
- a non-positive pivot anywhere is reported (DBAT_E_NOTSPD) and the call returns;
- x does not depend on how the tasks were spread over CTAs and launches.
Every test first asserts the structure (segments, padding, term counts, chains, chain queue) it was built for.
"""
import copy
import os
from collections import defaultdict

import numpy as np
import pytest
import scipy.linalg as sla
import scipy.sparse as sp

pytestmark = pytest.mark.gpu

import dbat_b200
from dbat_b200 import _lib
from dbat_b200.synth import make_convergent_scene, make_scene
from oracle import lsa
from oracle.cameramodel import brown_euler_cam4
from oracle.dbatstruct import buildserialindices, buildweightmatrix, serialize

T = 64
EPS = np.finfo(float).eps
ETA_FACTOR = 10.0           # eta_dev <= max(ETA_FACTOR * eta_lapack, 2 sqrt(ld) eps)
FWD_RTOL = 1e-12            # x against LAPACK where cond(A) <= 1e4
PIVOT_RTOL = 1e-12          # min / max pivot against diag(chol(P A P')) where cond(A) <= 1e4
CHUNK = 10                  # terms per link of a partial-sum chain (TC_CHUNK in tilesym.cu)
DEFAULT_CHAIN_CTAS = 24     # DBAT_TC_CHAIN_CTAS unset (tchol_alloc)
ETA_RATIOS = []             # (eta_dev / eta_lapack, case) of every solve: printed at the end of the module


@pytest.fixture(scope='module', autouse=True)
def _built(built_lib):
    yield built_lib
    if ETA_RATIOS:
        r, case = max(ETA_RATIOS)
        print('\nlargest eta_dev / eta_lapack over %d solves: %.3g (%s)' % (len(ETA_RATIOS), r, case))


# ---------------------------------------------------------------------------------------------------------------
# matrices
# ---------------------------------------------------------------------------------------------------------------
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


def _grid_blocks(g, reach):
    """Co-visibility of a g x g block of images: every image coupled to its neighbours within `reach` grid steps."""
    idx = np.arange(g * g).reshape(g, g)
    return [(int(idx[i, j]), int(idx[k, l])) for i in range(g) for j in range(g)
            for k in range(max(0, i - reach), min(g, i + reach + 1)) for l in range(max(0, j - reach), min(g, j + reach + 1))
            if idx[k, l] < idx[i, j]]


def _graph(kind, rng):
    """Edges of a co-visibility graph: (number of images, list of pairs)."""
    if kind == 'band':                                   # a strip: every image overlaps the next three
        m = 300
        return m, [(i, j) for i in range(m) for j in range(i + 1, min(m, i + 4))]
    if kind == 'ring':                                   # a closed ring of stations
        m = 240
        return m, [(i, (i + d) % m) for i in range(m) for d in (1, 2)]
    if kind == 'grid':
        return 14 * 14, _grid_blocks(14, 1)
    if kind == 'geometric':                              # random geometric graph in the unit square
        m = 300
        p = rng.uniform(size=(m, 2))
        d = np.linalg.norm(p[:, None] - p[None], axis=2)
        i, j = np.nonzero(np.triu(d < 0.11, 1))
        return m, list(zip(i.tolist(), j.tolist()))
    if kind == 'long-band':
        m = 560
        return m, [(i, j) for i in range(m) for j in range(i + 1, min(m, i + 4))]
    raise ValueError(kind)


def _damped_free_network(kind, cond, seed):
    """kron(graph Laplacian, B) + lam I, B a random 6 x 6 SPD block: the normal matrix of a free network (a gauge
    freedom of six per component) under LM damping, lam chosen for the condition number `cond`."""
    rng = np.random.default_rng(seed)
    m, edges = _graph(kind, rng)
    Lg = np.zeros((m, m))
    for i, j in edges:
        Lg[i, j] = Lg[j, i] = -1.0
    Lg -= np.diag(Lg.sum(axis=1))
    G = rng.standard_normal((6, 6))
    B = G @ G.T + 0.5 * np.eye(6)
    A = np.kron(Lg, B)
    top = np.linalg.eigvalsh(Lg)[-1] * np.linalg.eigvalsh(B)[-1]
    lam = top / (cond - 1.0)
    return A + lam * np.eye(6 * m)


def _two_hub_spd(rng):
    """Block diagonal plus two hub blocks in tile columns 20 and 21 that every block couples to but that do not
    couple to each other: in the natural order, tile (21, 20) is fill with 20 terms, a partial-sum chain that must
    start from zero."""
    nb = 280
    h1, h2 = 215, 225                                    # columns 1290.., 1350..: tiles 20 and 21 of 27
    blocks = [(h, a) for a in range(213) for h in (h1, h2)]        # blocks 0..212 lie in tile columns 0..19
    return _banded_arrow_spd(6 * nb, 0, 0, rng, blocks=blocks)


# ---------------------------------------------------------------------------------------------------------------
# the device's order and structure, recovered on the host
# ---------------------------------------------------------------------------------------------------------------
def _symbolic(A, mode, leaf):
    """dbat_tile_symbolic on the co-visibility graph dbat_tile_chol_solve builds from A, plus the derived
    structure: x2s (S index of every column of A), perm (columns of A in elimination order), the elimination-tree
    parents of the tile columns and the chain-queue length."""
    n = A.shape[0]
    nImg = (n + 5) // 6
    r, c = np.nonzero(np.tril(A, -1))
    a, b = r // 6, c // 6
    pairs = np.unique(np.stack([a[a != b], b[a != b]], axis=1), axis=0) if len(r) else np.zeros((0, 2), np.int64)
    # one two-image point per coupled pair; a one-image point keeps the observation list non-empty
    img = np.concatenate([pairs.ravel(), [0]])
    op = np.concatenate([np.repeat(np.arange(len(pairs)), 2), [len(pairs)]])
    nEO = np.full(nImg, 6)
    nEO[-1] = n - 6 * (nImg - 1)
    sym = _lib.tile_symbolic(img, op, nImg, len(pairs) + 1, nEO, 0, mode=mode, leaf=leaf)
    sym['x2s'] = sym['imgS'][np.arange(n) // 6] + np.arange(n) % 6
    sym['perm'] = np.argsort(sym['x2s'])
    nT, tix = sym['nT'], sym['tix']
    parent = np.full(nT, -1)
    for J in range(nT - 1):
        below = np.flatnonzero(tix[J + 1:, J] >= 0)
        if len(below):
            parent[J] = J + 1 + below[0]
    sym['parent'] = parent
    I, J = sym['taskIJ'].T
    sym['nterm'] = np.diff(sym['termPtr'])
    # the chain queue (tilesym.cu): every final diagonal task and, per column, the final task of the tile in the row
    # of its elimination-tree parent.  One part: phase 1 is empty and this is the whole chain queue of phase 2.
    sym['chain_len'] = int(((sym['taskMode'] == 0) & ((I == J) | (I == parent[J]))).sum())
    kind = sym['s2kind']
    assert (kind == 1).sum() == n and kind[-1] == 2 and (kind == 2).sum() == 1
    assert np.array_equal(np.sort(sym['x2s']), np.flatnonzero(kind == 1))
    return sym


def _chains(sym):
    """Per tile: the number of terms of each of its tasks in list order (one entry: no chain)."""
    links = defaultdict(list)
    for (I, J), k in zip(sym['taskIJ'], sym['nterm']):
        links[(int(I), int(J))].append(int(k))
    return links


# ---------------------------------------------------------------------------------------------------------------
# criteria
# ---------------------------------------------------------------------------------------------------------------
def _eta(A, x, b):
    """Normwise backward error, the residual in long double."""
    r = b.astype(np.longdouble) - A.astype(np.longdouble) @ x.astype(np.longdouble)
    return float(np.abs(r).max() / (np.abs(A).sum(axis=1).max() * np.abs(x).max() + np.abs(b).max()))


def _reference(A, b, sym):
    """LAPACK's solution and the pivots diag(chol(P A P')) in the device's elimination order."""
    p = sym['perm']
    c, low = sla.cho_factor(A[np.ix_(p, p)], lower=True)
    x = np.empty_like(b)
    x[p] = sla.cho_solve((c, low), b[p])
    return x, np.diag(c).copy()


def _tile_solve(A, b, mode, leaf=40, repeat=1):
    x, st = _lib.tile_chol_solve(A, b, mode=mode, leaf=leaf, repeat=repeat)
    return x, st


def _check(A, b, mode, leaf, sym, case, wellcond, repeat=1):
    """One device solve against the reference; returns x."""
    x, st = _tile_solve(A, b, mode, leaf, repeat)
    assert st['rc'] == 0, case
    for k in ('nT', 'nSlots', 'nTasks', 'nTerms', 'depth'):
        assert int(st[k]) == sym[k], (case, k)
    assert np.all(np.isfinite(x)), case
    xr, piv = _reference(A, b, sym)
    eta_d, eta_l = _eta(A, x, b), _eta(A, xr, b)
    ETA_RATIOS.append((eta_d / max(eta_l, 1e-300), case))
    bound = max(ETA_FACTOR * eta_l, 2 * np.sqrt(sym['ld']) * EPS)
    assert eta_d <= bound, '%s: backward error %.3g, LAPACK %.3g' % (case, eta_d, eta_l)
    if wellcond:
        np.testing.assert_allclose(x, xr, rtol=FWD_RTOL, atol=FWD_RTOL * np.abs(xr).max(), err_msg=case)
        np.testing.assert_allclose([st['min_pivot'], st['max_pivot']], [piv.min(), piv.max()], rtol=PIVOT_RTOL,
                                   err_msg=case)
    else:
        # the smallest pivot of an ill-conditioned system is known only to ~cond * eps relative to the largest;
        # the statistics must still come from the real unknowns alone
        assert piv.min() * (1 - 1e-3) <= st['min_pivot'] <= st['max_pivot'], case
        np.testing.assert_allclose(st['max_pivot'], piv.max(), rtol=1e-10, err_msg=case)
    return x


# ---------------------------------------------------------------------------------------------------------------
# banded arrows and a dissected grid
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('n,bw,border,mode', [(50, 50, 0, 0), (423, 423, 0, -1), (700, 90, 9, 0), (2500, 200, 9, 1),
                                              (2500, 200, 9, 2), (6002, 600, 9, 2)])
def test_tile_cholesky_solver(n, bw, border, mode):
    """The sparse tile Cholesky on its own (ordering + symbolic analysis + persistent data-flow kernel +
    backward substitution) against LAPACK on matrices shaped like reduced camera systems."""
    rng = np.random.default_rng(n + mode)
    A = _banded_arrow_spd(n, bw, border, rng)
    b = rng.standard_normal(n)
    sym = _symbolic(A, mode, 40)
    x = _check(A, b, mode, 40, sym, 'arrow n=%d mode %d' % (n, mode), wellcond=True)
    x2, _ = _tile_solve(A, b, mode, 40, repeat=3)                # epochs: the flags are reused
    np.testing.assert_array_equal(x2, x)
    _, st3 = _tile_solve(A - 2 * np.diag(np.diag(A)), b, mode, 120)
    assert st3['rc'] == _lib.E_NOTSPD


def test_tile_cholesky_dissected_grid():
    """Co-visibility of a 2-D block of images (every image coupled to its neighbours within two grid steps):
    nested dissection gives independent subtrees; the factorisation must not care about the order."""
    rng = np.random.default_rng(4)
    A = _banded_arrow_spd(6 * 24 * 24, 0, 0, rng, blocks=_grid_blocks(24, 2))
    b = rng.standard_normal(A.shape[0])
    depth = {}
    for mode in (0, 1, 2):
        sym = _symbolic(A, mode, 40)
        _check(A, b, mode, 40, sym, 'grid 24 mode %d' % mode, wellcond=True)
        depth[mode] = sym['depth']
    assert depth[2] < depth[1]


# ---------------------------------------------------------------------------------------------------------------
# 1. real reduced camera systems
# ---------------------------------------------------------------------------------------------------------------
_RCS_CACHE = {}


def _reduced_camera_system(kind):
    """S = U - W V^-1 W' and its rhs from the oracle's weighted Jacobian at the start values, with the nine
    self-calibration IO columns moved last (a dense border, as in production).  Returns a function of lambda."""
    if kind in _RCS_CACHE:
        return _RCS_CACHE[kind]
    if kind == 'strip':
        s, _ = make_scene(300, 6000, rays=8, seed=5, build_indices=False)
    elif kind == 'strip-long':
        s, _ = make_scene(560, 8000, rays=8, seed=6, build_indices=False)
    else:
        rays = np.random.default_rng(9).integers(2, 60, 3000)
        s, _ = make_convergent_scene(160, 3000, rays, seed=9, build_indices=False)
    buildserialindices(s)
    x0 = serialize(s)
    n, nOP3 = len(x0), len(s.bundle.serial.OP.dest)
    nC, nIO = n - nOP3, len(s.bundle.serial.IO.dest)
    assert nIO == 9 and np.array_equal(s.bundle.serial.IO.dest, np.arange(9))
    r, J = brown_euler_cam4(x0, s, True)
    R = np.sqrt(buildweightmatrix(s))
    Jw = (sp.diags(R) @ J).tocsc()
    N = (Jw.T @ Jw).tocsc()
    g = -(Jw.T @ (R * r))
    U = N[:nC, :nC].toarray()
    Wc = N[:nC, nC:].tocsr()
    Vb = sp.bsr_matrix(N[nC:, nC:], blocksize=(3, 3))
    assert Vb.nnz == 3 * nOP3 and np.array_equal(Vb.indices, np.arange(nOP3 // 3))     # 3 x 3 point blocks
    Vblk = Vb.data
    lam0 = 1e-10 * N.diagonal().sum() / n                # lambda0 of levenberg_marquardt.m:88-106
    cam = np.r_[np.arange(nIO, nC), np.arange(nIO)]     # [EO; IO]

    def system(lam, jacobi):
        Vi = np.linalg.inv(Vblk + lam * np.eye(3))
        Vinv = sp.bsr_matrix((Vi, np.arange(nOP3 // 3), np.arange(nOP3 // 3 + 1)), shape=(nOP3, nOP3))
        WV = (Wc @ Vinv).tocsr()
        S = U + lam * np.eye(nC) - (WV @ Wc.T).toarray()
        rhs = g[:nC] - WV @ g[nC:]
        S, rhs = S[np.ix_(cam, cam)], rhs[cam]
        S = 0.5 * (S + S.T)
        if jacobi:                                        # with the diagonal of N + lambda I, as the step scales
            d = 1.0 / np.sqrt(U.diagonal()[cam] + lam)
            S, rhs = S * d[:, None] * d[None, :], rhs * d
        return S, rhs

    _RCS_CACHE[kind] = (system, lam0)
    return _RCS_CACHE[kind]


@pytest.mark.parametrize('kind', ['strip', 'rings'])
@pytest.mark.parametrize('damped', [False, True])
@pytest.mark.parametrize('jacobi', [False, True])
def test_reduced_camera_systems(kind, damped, jacobi):
    system, lam0 = _reduced_camera_system(kind)
    S, rhs = system(lam0 if damped else 0.0, jacobi)
    n = S.shape[0]
    assert np.all(S[-9:] != 0)                            # the IO border couples to every unknown
    depth = {}
    for mode in (0, 1, 2):
        sym = _symbolic(S, mode, 40)
        assert sym['nT'] * T == sym['ld'] and sym['ld'] >= n + 1
        if mode == 0:                                     # natural order: the border is eliminated last
            assert sym['x2s'][-9:].min() > sym['x2s'][:-9].max()
        depth[mode] = sym['depth']
        _check(S, rhs, mode, 40, sym, '%s lam=%s jacobi=%s mode %d' % (kind, damped, jacobi, mode), wellcond=False)
    assert depth[1] <= depth[0]


# ---------------------------------------------------------------------------------------------------------------
# 2. damped gauge-free systems, 3. scale spread
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('kind,mode', [('band', 1), ('ring', 2), ('grid', 2), ('geometric', 0)])
@pytest.mark.parametrize('cond', [1e4, 1e8, 1e12])
def test_damped_free_networks(kind, mode, cond):
    A = _damped_free_network(kind, cond, seed=int(np.log10(cond)))
    ev = np.linalg.eigvalsh(A)
    assert 0.5 * cond <= ev[-1] / ev[0] <= 2 * cond
    sym = _symbolic(A, mode, 40)
    if mode == 2:
        assert sym['nSeg'] > 1 and (sym['s2kind'][:sym['x2s'].max()] == 0).any()     # dissected, aligned segments
    b = np.random.default_rng(1).standard_normal(A.shape[0])
    _check(A, b, mode, 40, sym, '%s cond %g' % (kind, cond), wellcond=cond <= 1e4)


@pytest.mark.parametrize('kind,mode', [('ring', 2), ('geometric', 1)])
def test_scale_spread(kind, mode):
    """D A D with D log-uniform over 1e-6 .. 1e6: entries over 24 decades, every approximate reciprocal and square
    root far from 1."""
    rng = np.random.default_rng(3)
    A = _damped_free_network(kind, 1e8, seed=8)
    d = 10.0 ** rng.uniform(-6, 6, A.shape[0])
    A = A * d[:, None] * d[None, :]
    sym = _symbolic(A, mode, 40)
    b = rng.standard_normal(A.shape[0]) * d
    _check(A, b, mode, 40, sym, 'D A D %s' % kind, wellcond=False)


# ---------------------------------------------------------------------------------------------------------------
# 4. edge shapes
# ---------------------------------------------------------------------------------------------------------------
EDGE_N = [1, 5, 6, 7, 62, 63, 64, 65, 127, 128, 129, 383, 384, 385, 1535, 1536]


@pytest.mark.parametrize('n', EDGE_N)
def test_edge_shapes(n):
    """A well-conditioned band with an arrow border: n around the tile size and the 6-column blocks (the rhs row
    at the end of a tile, alone in a tile, ...), natural / RCM / nested-dissection order, dissection leaves of 4
    images (alignment padding everywhere) and of 40; 1535 / 1536 straddle the automatic mode's switch."""
    rng = np.random.default_rng(n)
    A = _banded_arrow_spd(n, min(n, 40), min(n // 3, 9), rng)
    b = rng.standard_normal(n)
    configs = [(0, 40), (1, 40), (2, 4), (2, 40)]
    if n in (1535, 1536):
        configs.append((-1, 40))
    for mode, leaf in configs:
        sym = _symbolic(A, mode, leaf)
        kind = sym['s2kind']
        assert sym['ld'] == sym['nT'] * T and sym['ld'] >= n + 1
        if mode in (0, 1) or sym['nSeg'] == 1:
            assert sym['ld'] == (n + 1 + T - 1) // T * T             # no alignment padding, only the tail
        if mode == 2 and leaf == 4 and n >= 129:
            assert sym['nSeg'] > 2 and (kind[:sym['x2s'].max()] == 0).sum() >= 64
        if mode == -1:
            assert sym['mode'] == (0 if n < 24 * T else 2)
        _check(A, b, mode, leaf, sym, 'n=%d mode %d leaf %d' % (n, mode, leaf), wellcond=True)


def test_scaled_pivot_statistics():
    """The same padding-heavy system scaled by 1e-8 and 1e+8: the statistics must move with the scale, so neither a
    padding pivot (1) nor the rhs row's (~1e150) may ever enter them."""
    rng = np.random.default_rng(11)
    n = 385
    A = _banded_arrow_spd(n, 40, 9, rng)
    b = rng.standard_normal(n)
    sym = _symbolic(A, 2, 4)
    assert (sym['s2kind'] == 0).sum() > 64
    x1 = _check(A, b, 2, 4, sym, 'unscaled', wellcond=True)
    for f in (1e-8, 1e8):
        x = _check(A * f, b * f, 2, 4, sym, 'scaled %g' % f, wellcond=True)
        np.testing.assert_allclose(x, x1, rtol=1e-12, atol=1e-12 * np.abs(x1).max())
        _, st = _tile_solve(A * f, b * f, 2, 4)
        assert st['max_pivot'] < 1e-2 if f < 1 else st['min_pivot'] > 1e2


@pytest.mark.parametrize('case', ['block-diagonal', 'two-bands', 'arrow-partial-border'])
def test_disconnected_and_bordered(case):
    rng = np.random.default_rng(len(case))
    if case == 'block-diagonal':                         # no coupling at all: every block its own component
        n = 400
        A = _banded_arrow_spd(n, 0, 0, rng, blocks=[])
        for k in range(0, n, 6):
            G = rng.standard_normal((min(6, n - k), min(6, n - k)))
            A[k:k + 6, k:k + 6] += G @ G.T
    elif case == 'two-bands':
        n1, n2 = 600, 540
        A = sla.block_diag(_banded_arrow_spd(n1, 30, 0, rng), _banded_arrow_spd(n2, 30, 0, rng))
    else:                                                # the dense border is exactly the last, partial block
        n = 6 * 120 + 3
        A = _banded_arrow_spd(n, 40, 3, rng)
    n = A.shape[0]
    b = rng.standard_normal(n)
    for mode, leaf in ((0, 40), (1, 40), (2, 4), (2, 40)):
        sym = _symbolic(A, mode, leaf)
        if case == 'block-diagonal':
            assert np.count_nonzero(A - np.diag(np.diag(A))) == 30 * ((n + 5) // 6 - 1) + 12    # 6 x 6 blocks only
            if mode == 2:                                # a tile per block, the rhs in the last one: terms only there
                assert sym['nSeg'] == (n + 5) // 6 == sym['nT']
                assert np.all(sym['nterm'][sym['taskIJ'][:, 0] < sym['nT'] - 1] == 0)
        if case == 'two-bands' and mode != 0:
            assert sym['nSeg'] >= 2
        if case == 'arrow-partial-border' and mode == 0:
            assert n % 6 == 3 and sym['x2s'][-3:].min() > sym['x2s'][:-3].max() - 6
        _check(A, b, mode, leaf, sym, '%s mode %d leaf %d' % (case, mode, leaf), wellcond=True)


# ---------------------------------------------------------------------------------------------------------------
# 5. partial-sum chains
# ---------------------------------------------------------------------------------------------------------------
def test_chains_dense():
    """A dense system of 28 tile columns in natural order: tiles with 0 .. 27 terms - single tasks up to 15 terms,
    2-link chains from 16 (24: no tiny last link of 4), 3-link chains from 25 (no link shorter than half a chunk)."""
    n = 64 * 28 - 1
    rng = np.random.default_rng(28)
    G = rng.standard_normal((n, n))
    A = G @ G.T / n + np.eye(n)
    b = rng.standard_normal(n)
    sym = _symbolic(A, 0, 40)
    assert sym['nT'] == 28 and (sym['s2kind'] == 0).sum() == 0
    links = _chains(sym)
    total = {t: sum(v) for t, v in links.items()}
    assert sorted(set(total.values())) == list(range(28))
    for t, v in links.items():
        assert total[t] == t[1]                          # every k < J contributes
        assert len(v) == (1 if t[1] <= CHUNK + CHUNK // 2 else 2 if t[1] < 2 * CHUNK + CHUNK // 2 else 3), (t, v)
        assert all(k >= CHUNK // 2 for k in v[1:]) and max(v) <= CHUNK + CHUNK // 2
    assert sym['chain_len'] == 2 * 28 - 1
    _check(A, b, 0, 40, sym, 'dense 1791', wellcond=True)


def test_chains_inside_the_tree():
    """Nested dissection of a 2-D block: separators with more than 15 terms below them give chains on tiles of the
    tree, not only in the rhs row."""
    rng = np.random.default_rng(4)
    A = _banded_arrow_spd(6 * 24 * 24, 0, 0, rng, blocks=_grid_blocks(24, 2))
    b = rng.standard_normal(A.shape[0])
    sym = _symbolic(A, 2, 40)
    nT = sym['nT']
    chained = [t for t, v in _chains(sym).items() if len(v) > 1]
    assert sym['nSeg'] > 2 and any(I < nT - 1 for I, J in chained)
    _check(A, b, 2, 40, sym, 'grid 24 mode 2', wellcond=True)


def test_chain_on_a_fill_tile():
    """A chain whose tile is fill (not in the pattern of S): its first link starts from zero, every later link
    from the partial sum the one before left in the tile."""
    rng = np.random.default_rng(21)
    A = _two_hub_spd(rng)
    b = rng.standard_normal(A.shape[0])
    sym = _symbolic(A, 0, 40)
    tix, I, J = sym['tix'], sym['taskIJ'][:, 0], sym['taskIJ'][:, 1]
    k = np.flatnonzero((I == 21) & (J == 20))
    assert tix[21, 20] >= sym['nTopS'] and len(k) == 2                 # fill, two links
    assert sym['taskInit'][k].tolist() == [0, 1] and sym['nterm'][k].sum() == 20
    _check(A, b, 0, 40, sym, 'two hubs', wellcond=True)


# ---------------------------------------------------------------------------------------------------------------
# failures
# ---------------------------------------------------------------------------------------------------------------
def _failure_system():
    """A 16 x 16 grid of images, dissected with leaves of 40: separator tiles and alignment padding."""
    rng = np.random.default_rng(16)
    A = _banded_arrow_spd(6 * 16 * 16, 0, 0, rng, blocks=_grid_blocks(16, 2))
    return A, rng.standard_normal(A.shape[0])


@pytest.mark.parametrize('where', ['first', 'separator', 'last', 'before-padding'])
def test_negative_pivot_is_reported(where):
    """A' = A - (L_kk^2 + delta) e_k e_k' in the device's order: exactly pivot k turns negative, no earlier one
    changes.  The call must return DBAT_E_NOTSPD; the same matrix with +delta must solve."""
    A, b = _failure_system()
    sym = _symbolic(A, 2, 40)
    kind, nT, parent = sym['s2kind'], sym['nT'], sym['parent']
    real = np.flatnonzero(kind == 1)
    assert sym['nSeg'] > 2
    if where == 'first':
        s = real[0]
    elif where == 'last':
        s = real[-1]
        assert s // T == nT - 1                                       # shares the last tile with the rhs row
    elif where == 'separator':
        nchild = np.bincount(parent[parent >= 0], minlength=nT)
        seps = [J for J in range(nT - 1) if nchild[J] >= 2]
        assert seps
        s = real[real // T == seps[0]][3]
    else:
        gap = real[np.flatnonzero(np.diff(real) > 1)]                 # followed by alignment padding
        assert len(gap)
        s = gap[len(gap) // 2]
    pos = int(np.searchsorted(real, s))
    col = int(sym['perm'][pos])
    _, piv = _reference(A, b, sym)
    delta = 0.25 * piv[pos] ** 2
    bad = A.copy()
    bad[col, col] -= piv[pos] ** 2 + delta
    x, st = _tile_solve(bad, b, 2, 40)
    assert st['rc'] == _lib.E_NOTSPD, where
    ok = A.copy()
    ok[col, col] -= piv[pos] ** 2 - delta
    _check(ok, b, 2, 40, sym, 'pivot %s shrunk' % where, wellcond=True)


def test_handle_recovers_after_a_failed_factorisation():
    """The no-datum camcal network (7-dimensional gauge freedom) at a small negative lambda: V + lambda I stays
    positive definite while S(lambda) is indefinite, so the step must report `singular`.  The next step on the same
    handle, at LM's lambda0, must equal a fresh handle's and the oracle's point-first solve."""
    from oracle.loaders import camcal_pm_struct
    G = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'camcalpm')
    s = camcal_pm_struct(os.path.join(G, 'camcal-pmexport.txt'), None, keep_loaded=True)
    buildserialindices(s)
    x0 = serialize(s)
    n, nOP3 = len(x0), len(s.bundle.serial.OP.dest)
    nC = n - nOP3
    r, J = brown_euler_cam4(x0, s, True)
    R = np.sqrt(buildweightmatrix(s))
    Jw = (sp.diags(R) @ J).tocsc()
    N = (Jw.T @ Jw).toarray()
    g = -(Jw.T @ (R * r))
    V = np.array([N[nC + 3 * i:nC + 3 * i + 3, nC + 3 * i:nC + 3 * i + 3] for i in range(nOP3 // 3)])
    assert np.count_nonzero(N[nC:, nC:]) == np.count_nonzero(sla.block_diag(*V))
    minV = np.linalg.eigvalsh(V).min()
    lam = -1e-3 * minV
    Vi = sla.block_diag(*np.linalg.inv(V + lam * np.eye(3)))
    S = N[:nC, :nC] + lam * np.eye(nC) - N[:nC, nC:] @ Vi @ N[nC:, :nC]
    ev = np.linalg.eigvalsh(0.5 * (S + S.T))
    assert minV + lam > 0 and (ev < 0.5 * lam).sum() == 7 and S.diagonal().min() > 0
    lam0 = 1e-10 * np.trace(N) / n
    P = dbat_b200.Problem(copy.deepcopy(s))
    try:
        _, st = P.normal_step(x0, lam, True)
        assert st['singular']
        p, st = P.normal_step(x0, lam0, False)
    finally:
        P.close()
    P2 = dbat_b200.Problem(copy.deepcopy(s))
    try:
        p2, st2 = P2.normal_step(x0, lam0, False)
    finally:
        P2.close()
    # camcal's points have up to 21 rays, so the Schur update takes the atomic per-point kernel above 20 rays and two
    # handles differ by ~3e-11 whatever ran before (measured on a B200, 1000 W): not bit-identical, but any tile
    # or flag left over from the failed factorisation would show far above 1e-9
    assert np.all(np.isfinite(p)) and np.max(np.abs(p - p2)) <= 1e-9 * np.max(np.abs(p2)), 'state left behind'
    po = lsa.solve_spd_pointfirst(sp.csc_matrix(N) + lam0 * sp.identity(n, format='csc'), g, nC)
    assert np.max(np.abs(p - po)) <= 5e-9 * np.max(np.abs(po))


# ---------------------------------------------------------------------------------------------------------------
# schedule independence
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('case', ['strip-long', 'long-band'])
def test_schedule_independence(case, monkeypatch):
    """Every task sums its terms in a fixed list order, so x is bit-identical whether the chain queue runs in the
    same launch as the bulk (DBAT_TC_CHAIN_CTAS=0), on one CTA of its own (=1: split once the chain queue has 4
    tasks) or on the default 24 (split from 96 tasks), and from one repetition to the next."""
    import torch
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    assert sms >= 4 * DEFAULT_CHAIN_CTAS                 # tchol_alloc keeps the default split on this device
    if case == 'strip-long':
        system, _ = _reduced_camera_system('strip-long')
        A, b = system(0.0, True)
        mode = 2
    else:
        A = _damped_free_network('long-band', 1e8, seed=2)
        b = np.random.default_rng(2).standard_normal(A.shape[0])
        mode = 1
    sym = _symbolic(A, mode, 40)
    assert sym['chain_len'] >= 4 * DEFAULT_CHAIN_CTAS     # default: split launch
    xs = {}
    for ctas in ('0', '1', None):
        if ctas is None:
            monkeypatch.delenv('DBAT_TC_CHAIN_CTAS', raising=False)
        else:
            monkeypatch.setenv('DBAT_TC_CHAIN_CTAS', ctas)
        xs[ctas] = _check(A, b, mode, 40, sym, '%s chain CTAs %s' % (case, ctas), wellcond=False)
        x2, _ = _tile_solve(A, b, mode, 40, repeat=2)
        assert np.array_equal(x2, xs[ctas]), 'repeat=2 differs (%s)' % ctas
    assert np.array_equal(xs['0'], xs['1']) and np.array_equal(xs['0'], xs[None])
