"""Seeded synthetic self-calibration scenes for BASELINE configs 4 and 5 (SURVEY.md §8d).

One physical camera (6000x4000 px, 4 um pixels, cc = 24 mm, Brown K1-3/P1-2, model 3),
`nImg` stations on a jittered grid over a square terrain patch, every object point seen by
its `rays` nearest stations whose projection falls inside the frame.  Observations are the
exact projections through the reference camera model (`res_euler_brown_1.m:81-97`, solved
for the pixel by fixed-point iteration) plus N(0, 0.5 px) noise.  Start values are the truth
perturbed as in the recipe; IO start is cc = 24.3, principal point at the sensor centre and
no distortion.  Datum: `seteoest(s,'depend',1)`.
"""
import numpy as np
from scipy.spatial import cKDTree

from .dbatstruct import new_struct, seteoest_depend, buildserialindices

SEED = 20240607
IM_W, IM_H, PX = 6000, 4000, 0.004
IO_TRUE = np.array([24.0, 12.02, -7.98, 1e-4, 0.0, 2e-4, -3e-7, 1e-10, -1e-5, 2e-5])
IO_START = np.array([24.3, 12.0, -8.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0])


def _rot(ang):
    """M = R1(omega) R2(phi) R3(kappa) for arrays of angles (3,N) → (N,3,3)."""
    sw, cw = np.sin(ang[0]), np.cos(ang[0])
    sp_, cp = np.sin(ang[1]), np.cos(ang[1])
    sk, ck = np.sin(ang[2]), np.cos(ang[2])
    M = np.empty((ang.shape[1], 3, 3))
    M[:, 0, 0] = cp * ck; M[:, 0, 1] = -cp * sk; M[:, 0, 2] = sp_
    M[:, 1, 0] = cw * sk + sw * sp_ * ck; M[:, 1, 1] = cw * ck - sw * sp_ * sk; M[:, 1, 2] = -sw * cp
    M[:, 2, 0] = sw * sk - cw * sp_ * ck; M[:, 2, 1] = sw * ck + cw * sp_ * sk; M[:, 2, 2] = cw * cp
    return M


def _ideal(Q, q0, M, f):
    """lhs = -f * pinhole(M'(Q-q0)) for paired arrays (N,3),(N,3),(N,3,3) → (N,2), depth."""
    X = Q - q0
    q = np.einsum('nrc,nr->nc', M, X)
    return -f * q[:, 0:2] / q[:, 2:3], q[:, 2]


def _pixel_from_ideal(l, io):
    """Solve lhs = brown(A (y - u0)) for the pixel u (model 3), fixed-point on a."""
    f, px, py, b1, b2 = io[0:5]
    Kt, Pt = -io[5:8], -io[8:10]
    a = l.copy()
    for _ in range(60):
        r2 = np.sum(a * a, axis=1)
        rad = Kt[0] * r2 + Kt[1] * r2 ** 2 + Kt[2] * r2 ** 3
        pTu = a @ Pt
        ts = Pt[None, :] * r2[:, None] + 2 * pTu[:, None] * a
        a_new = l - a * rad[:, None] - ts
        if np.max(np.abs(a_new - a)) < 1e-15:
            a = a_new
            break
        a = a_new
    x1 = a[:, 1]
    x0 = (a[:, 0] - b2 * x1) / (1 + b1)
    y0, y1 = x0 + px, x1 + py
    return np.stack([y0 / PX, -y1 / PX], axis=1)


def make_scene(nImg=1000, nOP=200000, rays=10, seed=SEED, noise_px=0.5, start_noise=1.0,
               build_indices=True, cache_dir=None):
    """Return a DBAT struct (start values) plus a dict with the ground truth.

    cache_dir: directory for a pickle of the generated scene (the generator is deterministic in
    its arguments; bench.py uses this so that repeated runs on one box skip the ~1 min of host work).
    """
    if cache_dir is not None:
        import os
        import pickle
        key = 'dbat_scene_%d_%d_%d_%d_%g_%g_%d.pkl' % (nImg, nOP, rays, seed, noise_px, start_noise, build_indices)
        path = os.path.join(cache_dir, key)
        if os.path.exists(path):
            with open(path, 'rb') as fh:
                return pickle.load(fh)
        out = make_scene(nImg, nOP, rays, seed, noise_px, start_noise, build_indices, None)
        try:
            with open(path + '.tmp%d' % os.getpid(), 'wb') as fh:
                pickle.dump(out, fh, protocol=4)
            os.replace(path + '.tmp%d' % os.getpid(), path)
        except OSError:
            pass
        return out
    rng = np.random.default_rng(seed)
    H = 110.0
    A_fp = (H * 24 / 24) * (H * 16 / 24)
    L = np.sqrt(nImg * A_fp / 12)
    g = int(np.ceil(np.sqrt(nImg)))
    gi, gj = np.meshgrid(np.arange(g), np.arange(g), indexing='ij')
    cells = np.stack([gi.ravel(), gj.ravel()], axis=1)[:nImg]
    edge = min(55.0, 0.2 * L)                          # stations stay inside the terrain patch
    cxy = edge + (cells + 0.5 + rng.uniform(-0.3, 0.3, cells.shape)) * ((L - 2 * edge) / g)
    EO = np.empty((6, nImg))
    EO[0:2] = cxy.T
    EO[2] = rng.uniform(80, 140, nImg)
    EO[3:5] = rng.normal(0, np.deg2rad(10), (2, nImg))
    for _ in range(100):                               # optical axis must hit the patch
        hit_x = EO[0] - EO[2] * np.tan(EO[4]) / np.cos(EO[3])
        hit_y = EO[1] + EO[2] * np.tan(EO[3])
        out = np.flatnonzero((hit_x < 0) | (hit_x > L) | (hit_y < 0) | (hit_y > L))
        if len(out) == 0:
            break
        EO[3:5, out] = rng.normal(0, np.deg2rad(10), (2, len(out)))
    EO[5] = rng.uniform(-np.pi, np.pi, nImg)
    M = _rot(EO[3:6])
    tree = cKDTree(cxy)
    kq = min(nImg, max(4 * rays, 48))

    def visible(Q):
        """(camera index, take mask) of the `rays` nearest stations that see each point."""
        n = Q.shape[0]
        idx = np.empty((n, kq), dtype=np.int64)
        take = np.zeros((n, kq), dtype=bool)
        for b0 in range(0, n, 100000):
            Qb = Q[b0:b0 + 100000]
            _, ib = tree.query(Qb[:, 0:2], k=kq)
            ib = ib.reshape(len(Qb), -1)
            ii = ib.ravel()
            l, depth = _ideal(np.repeat(Qb, kq, axis=0), EO[0:3, ii].T, M[ii], IO_TRUE[0])
            ok = (depth < 0) & (l[:, 0] > -11.9) & (l[:, 0] < 11.8) & (l[:, 1] > -7.9) & (l[:, 1] < 7.8)
            ok = ok.reshape(len(Qb), kq)
            idx[b0:b0 + 100000] = ib
            take[b0:b0 + 100000] = ok & (np.cumsum(ok, axis=1) <= rays)
        return idx, take

    def place():
        OP = np.empty((3, nOP))
        idx = np.empty((nOP, kq), dtype=np.int64)
        take = np.zeros((nOP, kq), dtype=bool)
        bad = np.arange(nOP)
        for _ in range(1000):                          # rejection sampling: exactly `rays` rays per point
            OP[0:2, bad] = rng.uniform(0, L, (2, len(bad)))
            OP[2, bad] = rng.uniform(0, 30, len(bad))
            idx[bad], take[bad] = visible(OP.T[bad])
            bad = bad[take[bad].sum(axis=1) < rays]
            if len(bad) == 0:
                return OP, idx, take
        raise RuntimeError('could not place all object points')

    min_obs = min(20, max(4, (rays * nOP) // (4 * nImg)))
    for attempt in range(8):                           # stations that end up starved look straight down
        OP, idx, take = place()
        cnt = np.bincount(idx[take], minlength=nImg)
        starved = np.flatnonzero(cnt < min_obs)
        if len(starved) == 0:
            break
        EO[3:5, starved] *= 0.25
        M = _rot(EO[3:6])
    else:
        raise RuntimeError('some stations see too few points')
    pj, slot = np.nonzero(take)
    ip_op = pj
    ip_img = idx[pj, slot]
    l, _ = _ideal(OP.T[ip_op], EO[0:3, ip_img].T, M[ip_img], IO_TRUE[0])
    uv = _pixel_from_ideal(l, IO_TRUE) + rng.normal(0, noise_px, (len(ip_op), 2))
    # start values
    EO0 = EO.copy()
    EO0[0:3] += start_noise * rng.normal(0, 0.05, (3, nImg))
    EO0[3:6] += start_noise * rng.normal(0, np.deg2rad(0.1), (3, nImg))
    OP0 = OP + start_noise * rng.normal(0, 0.1, OP.shape)
    s = new_struct(np.tile(IO_START[:, None], (1, nImg)), EO0, OP0, uv.T, ip_img, ip_op,
                   np.array([[PX], [PX]]), np.array([[IM_W], [IM_H]]), 3, 3, 2, noise_px)
    s.bundle.est.IO[:] = True
    s.bundle.est.IO[4, :] = False                      # setcamest(s,'all','not','sk')
    s.bundle.est.OP[:] = True
    seteoest_depend(s, 0)
    if build_indices:
        buildserialindices(s)
    truth = dict(IO=IO_TRUE.copy(), EO=EO, OP=OP, L=L)
    return s, truth


def _look_at_angles(d, kappa):
    """(omega, phi, kappa) of M = R1(omega) R2(phi) R3(kappa) whose camera looks along the unit vectors d (3,N):
    the camera's z axis, the third column of M, is -d (kappa turns the frame about it freely)."""
    return np.stack([np.arctan2(d[1], -d[2]), np.arcsin(np.clip(-d[0], -1, 1)), kappa])


def make_convergent_scene(nImg, nOP, ray_counts, seed=SEED, noise_px=0.5, start_noise=1.0, build_indices=True):
    """Seeded close-range convergent network around a 3-D object, with a caller-given ray count per point.

    Same camera, noise and start-value recipe as make_scene.  The stations sit on three rings around the x axis
    at elevations -15, 10 and 35 degrees (phi = the elevation, far from the gimbal lock of the omega-phi-kappa
    angles), 19-21 m from the centre, all looking at it with a random roll so that the principal point and the
    distortion stay well determined.  The object points fill a cylinder of radius 4 m and length 6 m about the
    same axis: every station sees all of it inside the 6000 x 4000 frame.  Point j is observed by the
    ray_counts[j] stations nearest to it in azimuth, so points close to each other have overlapping, contiguous
    image lists (which lets them share window Schur groups).  Datum: `seteoest(s,'depend',1)`.
    """
    ray_counts = np.asarray(ray_counts, dtype=np.int64)
    if ray_counts.shape != (nOP,) or ray_counts.min() < 1 or ray_counts.max() > nImg:
        raise ValueError('ray_counts must hold nOP counts in [1, nImg]')
    rng = np.random.default_rng(seed)
    nRing = 3
    ring = np.arange(nImg) % nRing
    elev = np.deg2rad(np.array([-15.0, 10.0, 35.0]))[ring]
    per = np.bincount(ring, minlength=nRing)
    az = np.empty(nImg)
    for r in range(nRing):                             # evenly spaced per ring, rings offset, jittered
        k = np.flatnonzero(ring == r)
        az[k] = 2 * np.pi * (np.arange(len(k)) + r / nRing + rng.uniform(-0.2, 0.2, len(k))) / per[r]
    az = np.mod(az, 2 * np.pi)
    D = rng.uniform(19.0, 21.0, nImg)
    q0 = D * np.stack([np.sin(elev), np.cos(elev) * np.cos(az), np.cos(elev) * np.sin(az)])
    EO = np.empty((6, nImg))
    EO[0:3] = q0
    EO[3:6] = _look_at_angles(-q0 / D, rng.uniform(-np.pi, np.pi, nImg))
    M = _rot(EO[3:6])
    paz = rng.uniform(0, 2 * np.pi, nOP)
    rho = np.sqrt(rng.uniform(0.0, 16.0, nOP))
    OP = np.stack([rng.uniform(-3.0, 3.0, nOP), rho * np.cos(paz), rho * np.sin(paz)])
    # the ray_counts[j] stations nearest in azimuth (circular distance; ties by station index)
    dist = np.abs(np.angle(np.exp(1j * (paz[:, None] - az[None, :]))))
    near = np.argsort(dist, axis=1, kind='stable')
    take = np.arange(nImg)[None, :] < ray_counts[:, None]
    ip_op = np.nonzero(take)[0]
    ip_img = near[take]
    l, depth = _ideal(OP.T[ip_op], EO[0:3, ip_img].T, M[ip_img], IO_TRUE[0])
    inside = (depth < 0) & (l[:, 0] > -11.9) & (l[:, 0] < 11.8) & (l[:, 1] > -7.9) & (l[:, 1] < 7.8)
    assert inside.all(), 'a station does not see the whole object volume'
    uv = _pixel_from_ideal(l, IO_TRUE) + rng.normal(0, noise_px, (len(ip_op), 2))
    EO0 = EO.copy()
    EO0[0:3] += start_noise * rng.normal(0, 0.05, (3, nImg))
    EO0[3:6] += start_noise * rng.normal(0, np.deg2rad(0.1), (3, nImg))
    OP0 = OP + start_noise * rng.normal(0, 0.1, OP.shape)
    s = new_struct(np.tile(IO_START[:, None], (1, nImg)), EO0, OP0, uv.T, ip_img, ip_op,
                   np.array([[PX], [PX]]), np.array([[IM_W], [IM_H]]), 3, 3, 2, noise_px)
    s.bundle.est.IO[:] = True
    s.bundle.est.IO[4, :] = False                      # setcamest(s,'all','not','sk')
    s.bundle.est.OP[:] = True
    seteoest_depend(s, 0)
    if build_indices:
        buildserialindices(s)
    truth = dict(IO=IO_TRUE.copy(), EO=EO, OP=OP)
    return s, truth


def make_scene_shard(nImg, nOP_total, rank, world, rays=10, seed=SEED, noise_px=0.5, start_noise=1.0):
    """One rank's share of a synthetic block for a point-sharded multi-GPU run: the stations (and their start
    values) are generated identically on every rank from `seed`; this rank's nOP_total/world object points, their
    observations and start values come from an independent stream (seed, rank).  Nothing of the whole block
    ever exists on one host.  Same recipe as make_scene (the station re-orientation pass for starved stations
    is replaced by a check: at the densities of BASELINE configs 4/5 it never triggers).

    Returns (s, truth) with s.OP / s.IP holding only this rank's points; x = [IO; EO; this rank's OP]."""
    rng = np.random.default_rng(seed)
    H = 110.0
    A_fp = (H * 24 / 24) * (H * 16 / 24)
    L = np.sqrt(nImg * A_fp / 12)
    g = int(np.ceil(np.sqrt(nImg)))
    gi, gj = np.meshgrid(np.arange(g), np.arange(g), indexing='ij')
    cells = np.stack([gi.ravel(), gj.ravel()], axis=1)[:nImg]
    edge = min(55.0, 0.2 * L)
    cxy = edge + (cells + 0.5 + rng.uniform(-0.3, 0.3, cells.shape)) * ((L - 2 * edge) / g)
    EO = np.empty((6, nImg))
    EO[0:2] = cxy.T
    EO[2] = rng.uniform(80, 140, nImg)
    EO[3:5] = rng.normal(0, np.deg2rad(10), (2, nImg))
    for _ in range(100):
        hit_x = EO[0] - EO[2] * np.tan(EO[4]) / np.cos(EO[3])
        hit_y = EO[1] + EO[2] * np.tan(EO[3])
        out = np.flatnonzero((hit_x < 0) | (hit_x > L) | (hit_y < 0) | (hit_y > L))
        if len(out) == 0:
            break
        EO[3:5, out] = rng.normal(0, np.deg2rad(10), (2, len(out)))
    EO[5] = rng.uniform(-np.pi, np.pi, nImg)
    EO0 = EO.copy()
    EO0[0:3] += start_noise * rng.normal(0, 0.05, (3, nImg))
    EO0[3:6] += start_noise * rng.normal(0, np.deg2rad(0.1), (3, nImg))
    M = _rot(EO[3:6])
    tree = cKDTree(cxy)
    kq = min(nImg, max(4 * rays, 48))
    lo, hi = (nOP_total * rank) // world, (nOP_total * (rank + 1)) // world
    nOP = hi - lo
    prng = np.random.default_rng([seed, 1 + rank, world])
    OP = np.empty((3, nOP))
    idx = np.empty((nOP, kq), dtype=np.int64)
    take = np.zeros((nOP, kq), dtype=bool)
    bad = np.arange(nOP)
    for _ in range(1000):
        OP[0:2, bad] = prng.uniform(0, L, (2, len(bad)))
        OP[2, bad] = prng.uniform(0, 30, len(bad))
        for b0 in range(0, len(bad), 100000):
            bb = bad[b0:b0 + 100000]
            Qb = OP.T[bb]
            _, ib = tree.query(Qb[:, 0:2], k=kq)
            ib = ib.reshape(len(Qb), -1)
            ii = ib.ravel()
            l, depth = _ideal(np.repeat(Qb, kq, axis=0), EO[0:3, ii].T, M[ii], IO_TRUE[0])
            ok = (depth < 0) & (l[:, 0] > -11.9) & (l[:, 0] < 11.8) & (l[:, 1] > -7.9) & (l[:, 1] < 7.8)
            ok = ok.reshape(len(Qb), kq)
            idx[bb] = ib
            take[bb] = ok & (np.cumsum(ok, axis=1) <= rays)
        bad = bad[take[bad].sum(axis=1) < rays]
        if len(bad) == 0:
            break
    else:
        raise RuntimeError('could not place all object points')
    pj, slot = np.nonzero(take)
    ip_img = idx[pj, slot]
    l, _ = _ideal(OP.T[pj], EO[0:3, ip_img].T, M[ip_img], IO_TRUE[0])
    uv = _pixel_from_ideal(l, IO_TRUE) + prng.normal(0, noise_px, (len(pj), 2))
    OP0 = OP + start_noise * prng.normal(0, 0.1, OP.shape)
    s = new_struct(np.tile(IO_START[:, None], (1, nImg)), EO0, OP0, uv.T, ip_img, pj,
                   np.array([[PX], [PX]]), np.array([[IM_W], [IM_H]]), 3, 3, 2, noise_px)
    s.bundle.est.IO[:] = True
    s.bundle.est.IO[4, :] = False
    s.bundle.est.OP[:] = True
    seteoest_depend(s, 0)
    buildserialindices(s)
    truth = dict(IO=IO_TRUE.copy(), EO=EO, OP=OP, L=L, op_range=(lo, hi))
    return s, truth
