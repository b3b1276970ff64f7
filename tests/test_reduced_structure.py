"""Structure of the reduced camera system S that the symbolic analysis (csrc/tilesym.cu) relies on, checked with
the host tools of tools/reduced_sparsity.py.

The block pattern of S is the co-visibility graph of the images, the graph the symbolic analysis orders.  With the
images in a bandwidth-reducing order and the shared IO block last, the Cholesky factor stays inside the band of that
pattern; with the IO block first it fills completely, which is why the symbolic analysis places it last."""
import os
import sys

import numpy as np
import scipy.sparse as sp
from scipy.sparse.csgraph import reverse_cuthill_mckee
from scipy.sparse.linalg import splu

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'tools'))


def test_band_of_the_reduced_system_survives_only_with_the_io_block_last():
    from dbat_b200.synth import make_scene
    from dbat_b200.dbatstruct import seteoest_depend
    from oracle.dbatstruct import buildserialindices, serialize, buildweightmatrix
    from oracle.cameramodel import brown_euler_cam4
    from reduced_sparsity import covisibility, symbolic_cholesky
    s, _ = make_scene(100, 4000, rays=8, seed=3, build_indices=False)
    seteoest_depend(s, 0)
    buildserialindices(s)
    x, W = serialize(s), buildweightmatrix(s)
    J = brown_euler_cam4(x, s, True)[1]
    Jw = (sp.diags(np.sqrt(W)) @ J).tocsc()
    N = (Jw.T @ Jw).tocsc()
    nIO, nEO = len(s.bundle.serial.IO.dest), len(s.bundle.serial.EO.dest)
    nC = nIO + nEO
    B = N[:nC, nC:]
    S = N[:nC, :nC].toarray() - (B @ splu(N[nC:, nC:].tocsc()).solve(B.T.toarray()))
    d = 1 / np.sqrt(np.diag(S))
    S = S * d[:, None] * d[None, :]
    nImg = s.EO.val.shape[1]
    eo_col = np.full(6 * nImg, -1)
    eo_col[s.bundle.serial.EO.src] = s.bundle.serial.EO.dest
    eo_col = eo_col.reshape(6, nImg, order='F')
    # (1) the EO x EO block pattern of S is the co-visibility graph
    G = covisibility(np.asarray(s.IP.img), np.asarray(s.IP.op), nImg)
    img_of = np.full(nC, -1)
    for i in range(nImg):
        img_of[eo_col[:, i][eo_col[:, i] >= 0]] = i
    r, c = np.nonzero(np.abs(S) > 1e-13)
    both = (img_of[r] >= 0) & (img_of[c] >= 0)
    pat = sp.csr_matrix((np.ones(both.sum()), (img_of[r[both]], img_of[c[both]])), shape=(nImg, nImg)).astype(bool)
    free = np.flatnonzero((eo_col >= 0).any(axis=0))              # the datum camera has no columns in S
    assert (pat[free][:, free] != G[free][:, free]).nnz == 0 and pat.nnz == G[free][:, free].nnz
    # (2) RCM image order, IO last: the factor's EO part stays inside the band of the pattern
    perm = np.asarray(reverse_cuthill_mckee(G.tocsr(), symmetric_mode=True))
    inv = np.empty(nImg, int)
    inv[perm] = np.arange(nImg)
    coo = G.tocoo()
    band = int(np.abs(inv[coo.row] - inv[coo.col]).max())
    assert band < nImg // 2
    order = np.array([k for i in perm for k in eo_col[:, i] if k >= 0] + list(s.bundle.serial.IO.dest))
    L = np.linalg.cholesky(S[np.ix_(order, order)])
    i, j = np.nonzero(np.abs(L[:nEO, :nEO]) > 1e-13)
    assert (i - j).max() <= 6 * (band + 1) - 1
    # and the symbolic factorisation of the tool predicts a superset of the numerical fill
    cnt = symbolic_cholesky(G, perm)
    blocks = {(inv[img_of[order[a]]], inv[img_of[order[b]]]) for a, b in zip(i, j)}
    assert len({(a, b) for a, b in blocks if a > b}) <= cnt.sum()
    # (3) x order (IO first, today's layout of S): the arrowhead fills the whole factor
    L0 = np.linalg.cholesky(S)
    assert np.count_nonzero(np.abs(L0) > 1e-13) > 0.98 * nC * (nC + 1) / 2
