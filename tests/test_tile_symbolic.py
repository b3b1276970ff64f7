"""Host side of the sparse tile Cholesky (dbat_b200/csrc/tilesym.cu), checked on CPU.

The symbolic analysis (elimination order of the images, 64 x 64 tile pattern with fill, task list of the
data-flow factorisation) is executed here by a NumPy emulation of the device kernels' task semantics
(tilechol.cu): tasks are run one after the other in LIST ORDER, and every tile a task reads must already be
final - which is exactly the property that makes the persistent kernel deadlock-free.  The result must be
the Cholesky factor of the permuted reduced system, and the backward substitution in `bwdCols` order must
solve it.
"""
import numpy as np
import pytest
import scipy.sparse as sp

from dbat_b200 import _lib
from dbat_b200.synth import make_scene

T = 64


def _reduced_pattern_matrix(s, sym, rng):
    """Random SPD matrix in S order with exactly the structure of the reduced camera system: 6 x 6 blocks of
    co-visible images, dense IO rows, identity at padding positions."""
    nImg = s.EO.val.shape[1]
    ld = sym['ld']
    nEO = s.bundle.est.EO[:6].sum(axis=0).astype(int)
    A = sp.csr_matrix((np.ones(len(s.IP.img)), (s.IP.op, s.IP.img)))
    G = (A.T @ A).tocoo()
    S = np.zeros((ld, ld))
    for a, b in zip(G.row, G.col):
        if nEO[a] == 0 or nEO[b] == 0:
            continue
        ra = slice(sym['imgS'][a], sym['imgS'][a] + nEO[a])
        rb = slice(sym['imgS'][b], sym['imgS'][b] + nEO[b])
        S[ra, rb] = rng.normal(size=(nEO[a], nEO[b]))
    kind = sym['s2kind']
    io = np.arange(sym['ioS'], sym['ioS'] + 9)
    S[io, :] = rng.normal(size=(9, ld)) * (kind == 1)[None, :]
    S = np.tril(S) + np.tril(S, -1).T
    S[kind != 1, :] = 0
    S[:, kind != 1] = 0
    S += np.diag(np.abs(S).sum(axis=1) + 1.0)            # diagonally dominant => SPD (padding: identity)
    return S


def _emulate(sym, S, rhs):
    nT, ld = sym['nT'], sym['ld']
    tix = sym['tix']
    M = S.copy()
    M[ld - 1, :] = rhs                                     # tchol_put_rhs
    M[ld - 1, ld - 1] = 1e300
    tiles, done = {}, set()
    # every entry of the lower triangle must lie in a stored tile
    r, c = np.nonzero(np.tril(M))
    assert np.all(tix[r // T, c // T] >= 0)
    aux = set()
    cur = {}                                               # tiles under accumulation (chains of partial sums)
    for k, ((I, J), t0, t1) in enumerate(zip(sym['taskIJ'], sym['termPtr'][:-1], sym['termPtr'][1:])):
        slot = tix[I, J]
        assert slot >= 0 and slot not in done
        inS = slot < sym['nTopS'] or sym['nTop'] <= slot < sym['nTop'] + sym['nOwnS']
        if not inS:
            assert not M[I * T:(I + 1) * T, J * T:(J + 1) * T].any()      # a fill tile holds no entry of S
        if sym['taskWait'][k] >= 0:
            assert sym['taskWait'][k] in aux, 'chain link before its predecessor'
        if sym['taskInit'][k]:
            C = cur.get(slot, M[I * T:(I + 1) * T, J * T:(J + 1) * T]).copy()
            assert inS or slot in cur
        else:
            assert not inS and slot not in cur
            C = np.zeros((T, T))
        for a, b in sym['termAB'][t0:t1]:
            assert a in done and b in done, 'task list is not a topological order'
            C -= tiles[a] @ tiles[b].T
        if sym['taskMode'][k] == 1:
            cur[slot] = C
            if sym['taskSet'][k] >= 0:
                aux.add(int(sym['taskSet'][k]))
            continue
        if I == J:
            tiles[slot] = np.linalg.cholesky(np.tril(C) + np.tril(C, -1).T)
        else:
            d = tix[J, J]
            assert d in done
            tiles[slot] = np.linalg.solve(tiles[d], C.T).T
        done.add(slot)
    assert int((sym['taskMode'] == 0).sum()) == sym['nSlots']
    assert len(done) == sym['nSlots']
    L = np.zeros((ld, ld))
    for I in range(nT):
        for J in range(I + 1):
            if tix[I, J] >= 0:
                L[I * T:(I + 1) * T, J * T:(J + 1) * T] = tiles[tix[I, J]]
    # backward substitution in bwdCols order
    y = L[ld - 1, :].copy()
    y[ld - 1] = 0.0
    x = np.zeros(ld)
    xdone = set()
    for J in sym['bwdCols']:
        yj = y[J * T:(J + 1) * T].copy()
        for I in range(J + 1, nT):
            if tix[I, J] >= 0:
                assert I in xdone, 'bwdCols is not a valid order'
                xi = x[I * T:(I + 1) * T].copy()
                if I == nT - 1:
                    xi[T - 1] = 0.0
                yj -= tiles[tix[I, J]].T @ xi
        x[J * T:(J + 1) * T] = np.linalg.solve(tiles[tix[J, J]].T, yj)
        xdone.add(J)
    return L, x


@pytest.mark.parametrize('nImg,nOP,rays,mode', [(21, 100, 10, -1), (60, 900, 8, 1), (420, 9000, 8, 2), (420, 9000, 8, 1),
                                                (420, 9000, 8, 0)])
def test_task_list_factors_the_reduced_system(built_lib, nImg, nOP, rays, mode):
    s, _ = make_scene(nImg, nOP, rays=rays, seed=3, build_indices=False)
    nEO = s.bundle.est.EO[:6].sum(axis=0).astype(int)
    sym = _lib.tile_symbolic(s.IP.img, s.IP.op, nImg, nOP, nEO, 9, mode=mode, leaf=60)
    assert sym['nS'] == nEO.sum() + 9 and sym['ld'] % T == 0 and sym['ld'] > sym['ioS'] + 9
    assert (sym['s2kind'] == 1).sum() == sym['nS'] and sym['s2kind'][-1] == 2
    if mode == 2:
        assert sym['nSeg'] > 2 and sym['depth'] < sym['nT']        # independent subtrees shorten the chain
    rng = np.random.default_rng(5)
    S = _reduced_pattern_matrix(s, sym, rng)
    ld = sym['ld']
    rhs = rng.normal(size=ld) * (sym['s2kind'] == 1)
    L, x = _emulate(sym, S, rhs)
    n1 = ld - 1
    np.testing.assert_allclose(L[:n1, :n1] @ L[:n1, :n1].T, S[:n1, :n1], rtol=0, atol=1e-9 * np.abs(S).max())
    np.testing.assert_allclose(x[:n1], np.linalg.solve(S[:n1, :n1], rhs[:n1]), rtol=1e-9, atol=1e-12)


def test_orderings_are_permutations_and_dissection_shortens_the_chain(built_lib):
    s, _ = make_scene(600, 12000, rays=8, seed=11, build_indices=False)
    nEO = s.bundle.est.EO[:6].sum(axis=0).astype(int)
    res = {}
    for mode in (0, 1, 2):
        sym = _lib.tile_symbolic(s.IP.img, s.IP.op, 600, 12000, nEO, 9, mode=mode, leaf=60)
        used = np.sort(np.concatenate([np.arange(a, a + k) for a, k in zip(sym['imgS'], nEO) if k > 0]))
        assert len(np.unique(used)) == len(used) == nEO.sum()
        assert np.all(sym['s2kind'][used] == 1)
        res[mode] = sym
    assert res[2]['depth'] < 0.7 * res[1]['depth']
    assert res[1]['nTerms'] < res[0]['nTerms']                     # RCM beats the generator's order


@pytest.mark.parametrize('parts', [2, 4, 8])
def test_distributed_schedule_factors_the_reduced_system(built_lib, parts):
    """The factorisation cut into `parts` subtrees (tilesym.cu, nParts > 1), every part emulated in NumPy exactly as
    a rank runs it: phase 1 on its own columns plus partial sums into the separator ("top") tiles, the sum of the
    top tiles over the parts (the allreduce), phase 2 on the top columns everywhere, the backward substitution on
    top + own columns and the sum of the masked solutions.  Every read must hit a tile that is final ON THAT PART."""
    nImg, nOP = 700, 14000
    s, _ = make_scene(nImg, nOP, rays=8, seed=13, build_indices=False)
    nEO = s.bundle.est.EO[:6].sum(axis=0).astype(int)
    syms = [_lib.tile_symbolic(s.IP.img, s.IP.op, nImg, nOP, nEO, 9, mode=2, leaf=40, parts=parts, part=g) for g in range(parts)]
    sym = syms[0]
    assert sym['nParts'] == parts and (sym['colOwner'] >= 0).any() and (sym['colOwner'] < 0).any()
    for o in syms[1:]:                                              # everything but the task lists is identical
        for k in ('tix', 'imgS', 's2kind', 'colOwner', 'ownSBegin', 'ld', 'nTop', 'nTopS', 'nOwnS'):
            assert np.array_equal(o[k], sym[k]), k
    nT, ld, tix, owner = sym['nT'], sym['ld'], sym['tix'], sym['colOwner']
    rng = np.random.default_rng(8)
    S = _reduced_pattern_matrix(s, sym, rng)
    rhs = rng.normal(size=ld) * (sym['s2kind'] == 1)
    M = S.copy()
    M[ld - 1, :] = rhs
    M[ld - 1, ld - 1] = 1e300
    # every part starts from a random split of S (its "Schur contributions"); own tiles are reduced to the owner
    split = rng.dirichlet(np.ones(parts), size=1)[0]
    slotI = {int(tix[I, J]): (I, J) for I in range(nT) for J in range(I + 1) if tix[I, J] >= 0}

    def tile_of(A, slot):
        I, J = slotI[slot]
        return A[I * T:(I + 1) * T, J * T:(J + 1) * T]

    tiles = []                                                      # per part: slot -> array (current content)
    final = []                                                      # per part: slots holding final L values
    for g in range(parts):
        t = {}
        for slot in slotI:
            I, J = slotI[slot]
            inS = slot < sym['nTopS'] or sym['nTop'] <= slot < sym['nTop'] + sym['nOwnS']
            if owner[J] < 0:
                t[slot] = tile_of(M, slot) * split[g] if inS else np.zeros((T, T))     # local share of a top tile
            elif owner[J] == g:
                t[slot] = tile_of(M, slot).copy() if inS else np.zeros((T, T))         # after the reduce to the owner
        tiles.append(t)
        final.append(set())

    auxs = [set() for _ in range(parts)]

    def run(g, lo, hi, phase):
        sg, t, fin = syms[g], tiles[g], final[g]
        for k in range(lo, hi):
            I, J = sg['taskIJ'][k]
            slot = int(tix[I, J])
            mode = int(sg['taskMode'][k])
            if phase == 1:
                assert (owner[J] == g) or (owner[J] < 0 and mode == 1)
            else:
                assert owner[J] < 0
            if sg['taskWait'][k] >= 0:
                assert int(sg['taskWait'][k]) in auxs[g]
            C = t[slot].copy() if sg['taskInit'][k] else np.zeros((T, T))
            if not sg['taskInit'][k]:
                assert not t[slot].any()
            for a, b in sg['termAB'][sg['termPtr'][k]:sg['termPtr'][k + 1]]:
                assert int(a) in fin and int(b) in fin, 'read of a tile that is not final on this part'
                C -= t[int(a)] @ t[int(b)].T
            if mode == 1:
                t[slot] = C
                if sg['taskSet'][k] >= 0:
                    auxs[g].add(int(sg['taskSet'][k]))
                continue
            if I == J:
                t[slot] = np.linalg.cholesky(np.tril(C) + np.tril(C, -1).T)
            else:
                d = int(tix[J, J])
                assert d in fin
                t[slot] = np.linalg.solve(t[d], C.T).T
            fin.add(slot)

    for g in range(parts):
        run(g, 0, syms[g]['nTasks1'], 1)
    for slot in range(sym['nTop']):                                 # allreduce of the top tiles
        tot = sum(tiles[g][slot] for g in range(parts))
        for g in range(parts):
            tiles[g][slot] = tot.copy()
    for g in range(parts):
        run(g, syms[g]['nTasks1'], syms[g]['nTasks'], 2)
    # assemble L from the owners (top from part 0) and compare
    L = np.zeros((ld, ld))
    for slot, (I, J) in slotI.items():
        g = 0 if owner[J] < 0 else int(owner[J])
        assert slot in final[g]
        L[I * T:(I + 1) * T, J * T:(J + 1) * T] = tiles[g][slot]
    n1 = ld - 1
    np.testing.assert_allclose(L[:n1, :n1] @ L[:n1, :n1].T, S[:n1, :n1], rtol=0, atol=1e-9 * np.abs(S).max())
    # backward substitution per part, masked sum
    xsum = np.zeros(ld)
    for g in range(parts):
        t = tiles[g]
        x = np.zeros(ld)
        xdone = set()
        for J in syms[g]['bwdCols']:
            assert owner[J] < 0 or owner[J] == g
            yj = t[int(tix[nT - 1, J])][T - 1, :].copy()
            if J == nT - 1:
                yj[T - 1] = 0.0
            for I in range(J + 1, nT):
                if tix[I, J] >= 0:
                    assert I in xdone
                    xi = x[I * T:(I + 1) * T].copy()
                    if I == nT - 1:
                        xi[T - 1] = 0.0
                    yj -= t[int(tix[I, J])].T @ xi
            x[J * T:(J + 1) * T] = np.linalg.solve(t[int(tix[J, J])].T, yj)
            xdone.add(J)
        keep = np.repeat((owner == g) | ((owner < 0) & (g == 0)), T)
        xsum += x * keep
    np.testing.assert_allclose(xsum[:n1], np.linalg.solve(S[:n1, :n1], rhs[:n1]), rtol=1e-9, atol=1e-12)


@pytest.mark.parametrize('nImg,nOP', [(300, 20000), (1000, 40000)])
def test_distributed_analysis_keeps_the_image_order(built_lib, nImg, nOP):
    """The window Schur index is built at create from the one-part elimination order, and dbat_comm_init refuses a
    distributed analysis that orders the images with columns in S differently.  On synthetic blocks with a datum
    camera without columns, every part of a 2-, 4- or 8-part analysis keeps the one-part order."""
    s, _ = make_scene(nImg, nOP, rays=8, seed=17, build_indices=False)
    nEO = s.bundle.est.EO[:6].sum(axis=0).astype(int)
    assert (nEO == 0).any()
    has = np.flatnonzero(nEO > 0)

    def order(parts, part):
        sym = _lib.tile_symbolic(s.IP.img, s.IP.op, nImg, nOP, nEO, 9, parts=parts, part=part)
        assert sym['nParts'] == parts
        return has[np.argsort(sym['imgS'][has])]

    ref = order(1, 0)
    for parts in (2, 4, 8):
        for part in range(parts):
            assert np.array_equal(order(parts, part), ref), (parts, part)
