"""Host-side mirror of the reference's entry points for the bundle hot path.

Same names, argument meaning and return values as
`code/bundle/bundle.m`, `code/bundle/lsa/{levenberg_marquardt,levenberg_marquardt_powell,
gauss_newton_armijo}.m` and `code/bundle/bundle_cov.m`, with the per-iteration work done
by libdbatgpu.so (hand-written sm_100a kernels) through the C ABI in include/dbat_gpu.h.
The reference hands the optimisers an opaque closure `resFun=@(x)brown_euler_cam4(x,s)`
(`bundle.m:165`); here `resFun` is a `Problem` handle created from the same struct.
"""
import ctypes as C
import time
from types import SimpleNamespace as NS

import numpy as np
import scipy.sparse as sp

from . import _lib
from .dbatstruct import (buildserialindices, buildweightmatrix, column_matching, deserialize, paramtypes,
                         serialize)

_lin = lambda a: np.asarray(a).reshape(-1, order='F')


def covisibility_edges(img, op, nImg, nOP):
    """Pairs (a < b) of images that observe a common object point: the block pattern of the reduced camera system."""
    A = sp.csr_matrix((np.ones(len(img), dtype=np.int32), (np.asarray(op), np.asarray(img))), shape=(nOP, nImg))
    G = sp.triu((A.T @ A).tocsr(), 1).tocoo()
    return G.row.astype(np.int64), G.col.astype(np.int64)


class Problem:
    """Device-resident bundle problem: stands in for the closure `@(x)brown_euler_cam4(x,s)`.

    Calling it, `f = P(x)` / `f, J = P(x, True)`, evaluates the unweighted residual (and the
    sparse Jacobian) exactly like `[f,J]=feval(resFun,x)`.
    """

    def __init__(self, s, points=None, cam_priors=True, covis=None):
        """points=(lo,hi): keep only object points lo..hi-1 and their observations (one shard of
        a point-partitioned multi-GPU run; x stays the global vector).  cam_priors=False drops
        the IO/EO prior observations (they are counted on rank 0 only).  covis=(a, b): co-visibility edges
        (0-based image pairs) of the whole project when `s` itself holds only one rank's points."""
        if s.bundle.serial is None or s.bundle.deserial is None:
            buildserialindices(s)
        L = _lib.lib()
        dm = np.unique(s.IO.model.distModel)
        if len(dm) != 1:
            raise ValueError('Mixed lens distortion models not implemented.')   # brown_euler_cam4.m:30-33
        self.s = s
        ser, des = s.bundle.serial, s.bundle.deserial
        keep = {}
        d = _lib.ProblemDesc()
        nImg, nOP = s.EO.val.shape[1], s.OP.val.shape[1]
        lo, hi = (0, nOP) if points is None else points
        self.points = (lo, hi)
        sel = slice(None) if points is None else np.flatnonzero((s.IP.op >= lo) & (s.IP.op < hi))
        d.nImg, d.nOP = nImg, hi - lo
        d.nIP = len(s.IP.img) if points is None else len(sel)
        d.distModel, d.nK, d.nP = int(dm[0]), int(s.IO.model.nK), int(s.IO.model.nP)

        def put(name, arr, kind):
            a = _lib.f64(arr) if kind == 'd' else _lib.i64(arr)
            keep[name] = a
            setattr(d, name, _lib.dptr(a) if kind == 'd' else _lib.iptr(a))

        put('IOval', _lin(s.IO.val), 'd')
        put('EOval', _lin(s.EO.val[0:6]), 'd')
        put('OPval', _lin(s.OP.val[:, lo:hi]), 'd')
        put('IPval', _lin(s.IP.val[:, sel]), 'd')
        put('IPstd', _lin(s.IP.std[:, sel]), 'd')
        put('IPimg', s.IP.img[sel] + 1, 'i')
        put('IPop', s.IP.op[sel] - lo + 1, 'i')
        put('pxSize', _lin(s.IO.sensor.pxSize), 'd')
        d.n = ser.n
        for nm in ('IO', 'EO', 'OP'):
            dd = getattr(des, nm)
            src, dest = dd.src, dd.dest
            if nm == 'OP' and points is not None:
                k = (dest >= 3 * lo) & (dest < 3 * hi)
                src, dest = src[k], dest[k] - 3 * lo
            put(nm + 'des_src', src + 1, 'i')
            put(nm + 'des_dest', dest + 1, 'i')
            setattr(d, 'n%sdes' % nm, len(src))
        px, pv, ps = [], [], []
        for nm in ('IO', 'EO', 'OP'):                      # prior_obs.m:28-65, buildweightmatrix.m:26-31
            sr, pr = getattr(ser, nm), getattr(s.prior, nm)
            xi = sr.dest[sr.obs] + 1
            vv = _lin(pr.val)[sr.src[sr.obs]]
            sd = _lin(pr.std)[_lin(pr.use)]
            if nm == 'OP' and points is not None:
                k = (sr.src[sr.obs] >= 3 * lo) & (sr.src[sr.obs] < 3 * hi)
                xi, vv, sd = xi[k], vv[k], sd[k]
            if nm != 'OP' and not cam_priors:
                xi, vv, sd = xi[:0], vv[:0], sd[:0]
            px.append(xi); pv.append(vv); ps.append(sd)
            setattr(d, 'nPrior' + nm, len(xi))
        put('prior_x', np.concatenate(px), 'i')
        put('prior_val', np.concatenate(pv), 'd')
        put('prior_std', np.concatenate(ps), 'd')
        d.nCovis = 0
        if points is not None or covis is not None:
            # every rank must order and tile the reduced camera system identically: hand the library the
            # co-visibility graph of the whole project, not only of this shard's points
            ca, cb = covis if covis is not None else covisibility_edges(s.IP.img, s.IP.op, nImg, nOP)
            put('covis_a', np.asarray(ca) + 1, 'i')
            put('covis_b', np.asarray(cb) + 1, 'i')
            d.nCovis = len(ca)
        h = C.c_void_p()
        rc = L.dbat_create(C.byref(d), C.byref(h))
        if rc != 0:
            raise _lib.DbatError(rc, L.dbat_last_error(None).decode())
        self._h = h
        self.n = int(L.dbat_num_unknowns(h))
        self.m = int(L.dbat_num_residuals(h))
        self.last_phase = {}

    # -- lifetime
    def close(self):
        if getattr(self, '_h', None):
            _lib.lib().dbat_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != 0:
            raise _lib.DbatError(rc, _lib.lib().dbat_last_error(self._h).decode())

    # -- [f,J]=feval(resFun,x)
    def __call__(self, x, want_jac=False, weighted=False):
        x = _lib.f64(x)
        r = np.empty(self.m)
        self._check(_lib.lib().dbat_eval(self._h, _lib.dptr(x), _lib.dptr(r), int(weighted)))
        if not want_jac:
            return r
        return r, self.jacobian(weighted)

    def jacobian(self, weighted=False):
        """Sparse Jacobian (CSC, exact zeros dropped) at the x of the last eval/solve."""
        L = _lib.lib()
        nnz = C.c_int64()
        self._check(L.dbat_jacobian_nnz(self._h, int(weighted), C.byref(nnz)))
        Jc = np.empty(self.n + 1, dtype=np.int64)
        Ir = np.empty(max(1, nnz.value), dtype=np.int64)
        V = np.empty(max(1, nnz.value))
        self._check(L.dbat_jacobian_csc(self._h, int(weighted), _lib.iptr(Jc), _lib.iptr(Ir),
                                        _lib.dptr(V)))
        return sp.csc_matrix((V[:nnz.value], Ir[:nnz.value], Jc), shape=(self.m, self.n))

    def normal_step(self, x=None, lam=0.0, jacobi=False, trial=False, accept=False, p_out=None,
                    want_p=True):
        """One pass of the hot path (eval + assembly + Schur + Cholesky + back-substitution
        [+ trial residual]).  x=None reuses the device-resident iterate."""
        xa = _lib.f64(x) if x is not None else None
        p = p_out if p_out is not None else (np.empty(self.n) if want_p else None)
        st = np.zeros(8)
        flags = int(jacobi) | (2 if trial else 0) | (4 if accept else 0)
        self._check(_lib.lib().dbat_normal_step(self._h, _lib.dptr(xa), float(lam), flags,
                                                _lib.dptr(p), _lib.dptr(st)))
        return p, dict(f=st[0], jp2=st[1], rjp=st[2], singular=bool(st[3]), launches=int(st[4]),
                       f_new=st[5], device_ms=st[6])

    def set_devices(self, devices):
        """One process, several GPUs (dbat_set_devices): shard this problem's object points over the listed CUDA
        devices.  Every later call on the handle runs on all of them and returns merged results."""
        arr = (C.c_int * len(devices))(*[int(d) for d in devices])
        self._check(_lib.lib().dbat_set_devices(self._h, arr, len(devices)))
        return self

    def reduced_info(self):
        """Structure of the reduced camera system (tile counts, factorisation work, chain depth) and the point-side
        paths the problem takes (points over 128 rays, points over 20 rays, largest group union and group size)."""
        v = np.zeros(16, dtype=np.int64)
        self._check(_lib.lib().dbat_reduced_info(self._h, _lib.iptr(v)))
        names = ['nT', 'ld', 'nS', 'nSlots', 'nSlotsS', 'nTasks', 'nTerms', 'depth', 'order_mode', 'nSeg', 'gridFactor', 'gridBwd',
                 'nPsbig', 'nBig', 'grpMaxRays', 'grpMaxPts']
        d = {k: int(v[i]) for i, k in enumerate(names)}
        d['flops'] = 2.0 * 64 ** 3 * d['nTerms'] + 64.0 ** 3 * (d['nSlots'] - d['nT']) + d['nT'] * 64.0 ** 3 / 3
        return d

    def phase_times(self):
        names = (C.c_char_p * 16)()
        ms = np.zeros(16)
        cnt = np.zeros(16, dtype=np.int64)
        k = _lib.lib().dbat_phase_times(self._h, names, _lib.dptr(ms), _lib.iptr(cnt), 16)
        return {names[i].decode(): (float(ms[i]), int(cnt[i])) for i in range(k)}

    def solve(self, method, x0, maxIter=20, convTol=1e-6, absTerm=False, doTrace=False,
              singularTest=True, want_trace=True, want_resid=True, **kw):
        L = _lib.lib()
        o = _lib.Opts()
        L.dbat_default_opts(_lib.METHOD[method], C.byref(o))
        o.maxIter, o.convTol, o.absTerm = int(maxIter), float(convTol), int(absTerm)
        o.doTrace, o.singularTest = int(doTrace), int(singularTest)
        for k, v in kw.items():
            if v is not None:
                setattr(o, k, v)
        cap = int(maxIter) + 2
        x0 = _lib.f64(x0)
        bufs = dict(x=np.empty(self.n), p=np.empty(self.n), rr=np.full(cap + 1, np.nan),
                    damping=np.full(cap + 1, np.nan), rhos=np.full(cap, np.nan),
                    steps=np.zeros(cap, dtype=np.int32))
        if want_resid:
            bufs['r_w'] = np.empty(self.m)
            bufs['r_u'] = np.empty(self.m)
        if want_trace:
            bufs['trace'] = np.full((cap, self.n), np.nan)     # row = one x (column of T)
        res = _lib.Result()
        for k in ('x', 'p', 'rr', 'damping', 'rhos', 'r_w', 'r_u', 'trace'):
            setattr(res, k, _lib.dptr(bufs[k]) if k in bufs else None)
        res.steps = bufs['steps'].ctypes.data_as(C.POINTER(C.c_int32))
        self._check(L.dbat_solve(self._h, _lib.METHOD[method], C.byref(o), _lib.dptr(x0), C.byref(res)))
        out = NS(x=bufs['x'], code=int(res.code), n=int(res.iters), p=bufs['p'],
                 rr=bufs['rr'][:res.nRr].copy(), damping=bufs['damping'][:res.nDamping].copy(),
                 rhos=bufs['rhos'][:res.nRhos].copy(), steps=bufs['steps'][:res.nDamping].copy(),
                 T=bufs['trace'][:res.nTrace].T.copy() if want_trace else None,
                 r_w=bufs.get('r_w'), r_u=bufs.get('r_u'),
                 seconds=float(res.seconds), launches=int(res.launches))
        self.last_phase = self.phase_times()
        return out

    def cov_stats(self, s0, thres=0.95):
        """Report-side consumers of the posterior covariance, computed on the device from one factorisation
        (`dbat_cov_stats`; bundle_result_file.m:92-153, corrmat.m, high_{io,eo,op}_correlations.m in block form).
        Returns a dict: 'std' (n, x order) and 'io' / 'eo' / 'op' = (row, col, block, rho) arrays of the pairs with
        |correlation| > thres, 0-based, in the reference's order (block, then column, then row).  After a failed
        factorisation the deviations are NaN and the lists empty."""
        L = _lib.lib()
        s = self.s
        nImg, nOP, NC = s.EO.val.shape[1], s.OP.val.shape[1], s.IO.val.shape[0]
        std = np.zeros(self.n)
        caps = {'io': nImg * NC * (NC - 1) // 2, 'eo': nImg * 15, 'op': nOP * 3}
        lists, keep = {}, {}
        for k, cap in caps.items():
            cap = max(1, cap)
            arr = (np.zeros(cap, dtype=np.int64), np.zeros(cap, dtype=np.int32), np.zeros(cap, dtype=np.int32), np.zeros(cap))
            keep[k] = arr
            lists[k] = _lib.CovHitList(cap, 0, arr[0].ctypes.data_as(C.POINTER(C.c_int64)), arr[1].ctypes.data_as(C.POINTER(C.c_int32)),
                                       arr[2].ctypes.data_as(C.POINTER(C.c_int32)), arr[3].ctypes.data_as(C.POINTER(C.c_double)))
        rc = L.dbat_cov_stats(self._h, float(s0), float(thres), _lib.dptr(std), C.byref(lists['io']), C.byref(lists['eo']), C.byref(lists['op']))
        if rc not in (0, _lib.E_NOTSPD):
            self._check(rc)
        out = {'std': std, 'failed': rc != 0}
        for k in caps:
            m = 0 if rc else int(min(lists[k].n, lists[k].cap))
            b, r, c, v = keep[k]
            out[k] = (r[:m].astype(np.int64), c[:m].astype(np.int64), b[:m].copy(), v[:m].copy())
        return out

    def cov(self, which, s0):
        L = _lib.lib()
        s = self.s
        nImg, nOP, NC = s.EO.val.shape[1], s.OP.val.shape[1], s.IO.val.shape[0]
        w = which.lower()
        if w == 'cio':
            out = np.zeros((nImg, NC, NC))
        elif w == 'ceo':
            out = np.zeros((nImg, 6, 6))
        elif w == 'cop':
            out = np.zeros((nOP, 3, 3))
        elif w == 'cxx_cam':
            nC = self.n - len(s.bundle.serial.OP.dest)
            out = np.zeros((nC, nC))
        elif w == 'cxx':
            out = np.zeros((self.n, self.n))
        elif w == 'cxx_op':
            m3 = len(s.bundle.serial.OP.dest)
            out = np.zeros((m3, m3))
        else:
            raise ValueError(which)
        rc = L.dbat_cov(self._h, _lib.COV[w], float(s0), _lib.dptr(out))
        if rc != _lib.E_NOTSPD:          # a failed factorisation is an outcome (NaN deviations), not an API error
            self._check(rc)
        if rc == _lib.E_NOTSPD or not np.isfinite(out).all():
            # the factorisation broke down (singular or NaN normal matrix): the reference then reports NaN
            # for every estimated element (bundle_cov.m:101-107,136-160), not a partly finite matrix
            out[out != 0] = np.nan
        return out


class _Final:
    """`final` struct of the optimisers (levenberg_marquardt.m:231-235); J is exported lazily."""

    def __init__(self, problem, r_u, r_w, p):
        self._problem = problem
        self.p = p
        self.unweighted = _RJ(problem, r_u, False)
        self.weighted = _RJ(problem, r_w, True)
        self.factorized = None
        self._scaled = None

    @property
    def scaled(self):
        """gauss_newton_armijo.m:166-174,249: column scaling D = 1/||J(:,j)|| and J*diag(D)."""
        if self._scaled is None:
            J = self.weighted.J
            with np.errstate(divide='ignore'):
                D = 1.0 / np.sqrt(np.asarray(J.multiply(J).sum(axis=0)).ravel())
            self._scaled = NS(D=D, J=(J @ sp.diags(D)).tocsc())
        return self._scaled


class _RJ:
    def __init__(self, problem, r, weighted):
        self.r = r
        self._problem, self._weighted, self._J = problem, weighted, None

    @property
    def J(self):
        if self._J is None:
            self._J = self._problem.jacobian(self._weighted)
        return self._J


def make_termfun(convTol=1e-6, absTerm=False):
    """bundle.m:186-192: termination closure; carries its constants for the device loop."""
    if absTerm:
        f = lambda Jp, r: np.linalg.norm(r) <= convTol
    else:
        f = lambda Jp, r: np.linalg.norm(Jp) <= convTol * np.linalg.norm(r)
    f.convTol, f.absTerm = convTol, absTerm
    return f


def _need_problem(resFun):
    if not isinstance(resFun, Problem):
        raise TypeError('resFun must be a dbat_b200.Problem handle; a plain residual function '
                        'belongs to the original (CPU) code path')
    return resFun


def _term_consts(termFun):
    if hasattr(termFun, 'convTol'):
        return termFun.convTol, termFun.absTerm
    raise TypeError('termFun must come from make_termfun(convTol, absTerm)')


def levenberg_marquardt(resFun, vetoFun, x0, W, maxIter, termFun, doTrace, lambda0, lambdaMin):
    """levenberg_marquardt.m:1-2: [x,code,n,final,T,rr,lambdas]."""
    P = _need_problem(resFun)
    if vetoFun:
        raise NotImplementedError('veto functions are undefined in the reference (bundle.m:169)')
    tol, absT = _term_consts(termFun)
    o = P.solve('lm', x0, maxIter, tol, absT, doTrace, lambda0=lambda0, lambdaMin=lambdaMin)
    final = _Final(P, o.r_u, o.r_w, o.p)
    P.last = o
    return o.x, o.code, o.n, final, o.T, o.rr, o.damping


def levenberg_marquardt_powell(resFun, vetoFun, x0, W, maxIter, termFun, doTrace, delta0, mu, eta):
    """levenberg_marquardt_powell.m:1-2: [x,code,n,final,T,rr,deltas,rhos,steps]."""
    P = _need_problem(resFun)
    if vetoFun:
        raise NotImplementedError('veto functions are undefined in the reference (bundle.m:169)')
    tol, absT = _term_consts(termFun)
    o = P.solve('lmp', x0, maxIter, tol, absT, doTrace, delta0=delta0, mu=mu, eta=eta)
    final = _Final(P, o.r_u, o.r_w, o.p)
    P.last = o
    return o.x, o.code, o.n, final, o.T, o.rr, o.damping, o.rhos, o.steps


def gauss_markov(resFun, x0, W, maxIter, convTol, trace, sTest):
    """gauss_markov.m:1: [x,code,n,final,T,rr]=gauss_markov(resFun,x0,W,maxIter,convTol,trace,sTest) -
    undamped Gauss-Newton with the relative termination test norm(J p) <= convTol norm(r).  (Through
    `bundle(s,'gm')` the reference passes a function handle as convTol, bundle.m:273, which fails; the
    direct call works and is what this mirrors.)"""
    P = _need_problem(resFun)
    o = P.solve('gm', x0, maxIter, float(convTol), False, trace, sTest)
    final = _Final(P, o.r_u, o.r_w, o.p)
    P.last = o
    return o.x, o.code, o.n, final, o.T, o.rr


def gauss_newton_armijo(resFun, vetoFun, x0, W, maxIter, termFun, trace, sTest, mu, alphaMin):
    """gauss_newton_armijo.m:1-2: [x,code,n,final,T,rr,alphas]."""
    P = _need_problem(resFun)
    if vetoFun:
        raise NotImplementedError('veto functions are undefined in the reference (bundle.m:169)')
    tol, absT = _term_consts(termFun)
    o = P.solve('gna', x0, maxIter, tol, absT, trace, sTest, mu=mu, alphaMin=alphaMin)
    final = _Final(P, o.r_u, o.r_w, o.p)
    P.last = o
    return o.x, o.code, o.n, final, o.T, o.rr, o.damping


VERSION = 'dbat_b200 0.1 (B200 device path)'


def bundle(s, *varargin):
    """bundle.m:1-76: [s,ok,iters,s0,E]=bundle(s[,maxIter|tol][,damping][,'trace'][,...])."""
    maxIter, damping, veto, singularTest = 20, 'gna', False, True      # bundle.m:78-87
    doTrace = dofVerb = pmDof = absTerm = False
    convTol = 1e-6
    for v in varargin:                                                 # bundle.m:88-132
        if isinstance(v, bool):
            veto = v
        elif isinstance(v, (int, float, np.integer, np.floating)):
            if v == round(v):
                maxIter = int(v)
            else:
                convTol = float(v)
        elif isinstance(v, str):
            lv = v.lower()
            if lv in ('none', 'gm', 'gna', 'lm', 'lmp'):
                damping = lv
            elif lv == 'trace':
                doTrace = True
            elif lv == 'singulartest':
                singularTest = True
            elif lv == 'nosingulartest':
                singularTest = False
            elif lv == 'pmdof':
                pmDof = True
            elif lv == 'dofverb':
                dofVerb = True
            elif lv == 'absterm':
                absTerm = True
            else:
                raise ValueError('DBAT:bundle:badInput Unknown damping')
        else:
            raise ValueError('DBAT:bundle:badInput Unknown parameter')
    for pri, est in ((s.prior.IO, s.bundle.est.IO), (s.prior.EO, s.bundle.est.EO),
                     (s.prior.OP, s.bundle.est.OP)):                   # bundle.m:137-154
        pri.use[~est] = False
    if s.bundle.serial is None or s.bundle.deserial is None:           # bundle.m:156-159
        buildserialindices(s)
    x0 = serialize(s)                                                  # bundle.m:162
    resFun = Problem(s)                                                # bundle.m:165
    vetoFun = None
    if veto:
        raise NotImplementedError('chirality veto is undefined in the reference (bundle.m:169)')
    W = buildweightmatrix(s)                                           # bundle.m:175
    termFun = make_termfun(convTol, absTerm)                           # bundle.m:186-192
    E = NS(maxIter=maxIter, convTol=convTol, absTerm=absTerm, singularTest=singularTest,
           chirality=veto, dateStamp=time.strftime('%d-%b-%Y %H:%M:%S'), version=VERSION)   # bundle.m:263-265
    t0 = time.process_time()
    if damping in ('none', 'gm'):
        raise NotImplementedError("'gm' is broken via bundle() in the reference (bundle.m:273-274)")
    elif damping == 'gna':                                             # bundle.m:275-295
        mu, alphaMin = 0.1, 1e-9
        x, code, iters, final, X, res, alpha = gauss_newton_armijo(
            resFun, vetoFun, x0, W, maxIter, termFun, doTrace, singularTest, mu, alphaMin)
        E.damping = NS(name='gna', alpha=alpha, mu=mu, alphaMin=alphaMin)
    elif damping == 'lm':                                              # bundle.m:296-315
        lambda0 = -1e-10
        x, code, iters, final, X, res, lam = levenberg_marquardt(
            resFun, vetoFun, x0, W, maxIter, termFun, doTrace, lambda0, lambda0)
        E.damping = NS(name='lm', **{'lambda': lam}, lambda0=lam[0], lambdaMin=lam[0])
    else:                                                              # bundle.m:316-335
        rhoBad, rhoGood = 0.25, 0.75
        delta0 = float(np.linalg.norm(x0))
        x, code, iters, final, X, res, delta, rho, step = levenberg_marquardt_powell(
            resFun, vetoFun, x0, W, maxIter, termFun, doTrace, delta0, rhoBad, rhoGood)
        E.damping = NS(name='lmp', delta=delta, rho=rho, delta0=delta0, rhoBad=rhoBad,
                       rhoGood=rhoGood, step=step)
    E.time = time.process_time() - t0
    E.gpu_seconds = resFun.last.seconds
    E.res, E.trace, E.code, E.usedIters, E.final = res, X, code, iters, final   # bundle.m:341-350
    E.problem = resFun
    E.x = x
    ok = code == 0
    if ok:                                                             # bundle.m:356-358
        deserialize(s, x)
        E.problem.s = s
    s.post.res.IP = final.unweighted.r[s.post.res.ix.IP].reshape(2, -1, order='F') \
        / s.IO.sensor.pxSize[:, s.IP.cam]                              # bundle.m:449-457
    p = 0
    if pmDof:                                                          # bundle.m:470-472
        seen_op = np.zeros(s.OP.val.shape[1], bool); seen_op[s.IP.op] = True
        seen_im = np.zeros(s.EO.val.shape[1], bool); seen_im[s.IP.img] = True
        p = np.count_nonzero(~s.bundle.est.OP[:, seen_op]) + \
            np.count_nonzero(~s.bundle.est.EO[0:6, seen_im])
    r = final.weighted.r                                               # bundle.m:476-491
    dof = len(r) + p - len(x)
    if dofVerb:
        print('bundle: dof=%d+%d-%d=%d.' % (len(r), p, len(x), dof))
    s0 = float(np.sqrt((r @ r) / dof))
    s.post.sigmas = s0 * s.IP.sigmas
    E.numObs, E.numParams, E.redundancy, E.s0, E.sigmas = len(r), len(x), dof, s0, s.post.sigmas
    E.paramTypes = paramtypes(s)                                       # bundle.m:162,368
    E.weakness = NS(structural=None, numerical=NS(rank=len(x), deficiency=0))
    if code in (-4, -2):
        # post-mortem diagnostics must not turn a reported failure code into an exception (the reference
        # wraps its rank estimate in try/catch as well, bundle.m:377-387): on error the ranks are NaN
        nan = float('nan')
        try:
            if code == -4:
                E.weakness = structural_weakness(final.weighted.J, E.paramTypes)
            else:
                E.weakness = NS(structural=None, numerical=numerical_weakness(final.scaled.J, E.paramTypes))
        except Exception as exc:                                       # noqa: BLE001
            E.weakness = NS(structural=NS(rank=nan, deficiency=nan, suspectedParams=[], error=repr(exc))
                            if code == -4 else None, numerical=NS(rank=nan, deficiency=nan, error=repr(exc)))
    return s, ok, iters, s0, E


def structural_weakness(J, paramTypes):
    """bundle.m:431-446: on code -4 record which parameters a maximum matching of the Jacobian's
    pattern leaves out (`dmperm`), the structural rank and its deficiency; the numerical rank is
    marked unchecked."""
    dm = column_matching(J)
    rank = int(np.count_nonzero(dm))
    return NS(structural=NS(dmperm=dm, rank=rank, deficiency=len(dm) - rank,
                            suspectedParams=list(np.asarray(paramTypes, dtype=object)[dm == 0])),
              numerical=NS(rank=float('nan'), deficiency=float('nan')))


NUMRANK_MAX_N = 6000       # dense SVD of the scaled Jacobian's Gram matrix; above it the rank is NaN


def numerical_weakness(Js, paramTypes):
    """bundle.m:373-428: on code -2, the numerical rank of the column-scaled Jacobian
    (spnrank.m:166-178: singular values above max(size)*eps(smax)), its deficiency and, when
    deficient, an orthonormal basis V of the null-space with eigenvalues d of Js'Js, trace (of the
    sqrt(eps)-shifted Js'Js, as the reference leaves it) and per vector the parameters whose
    entry exceeds the mean of the largest entry and sqrt(1/n).  A post-mortem diagnostic, done on the
    host like the reference's; beyond NUMRANK_MAX_N unknowns rank and deficiency are NaN, which is what
    the reference records when spnrank gives up (:384-387)."""
    m, n = Js.shape
    if n > NUMRANK_MAX_N:
        return NS(rank=float('nan'), deficiency=float('nan'))
    G = (Js.T @ Js).toarray()
    d, V = np.linalg.eigh(G)
    smax = np.sqrt(max(d[-1], 0.0))
    # singular values are sqrt(d), but squaring loses the small ones: re-measure ||Js v|| for every
    # eigenvector whose eigenvalue is within rounding of the squared tolerance
    tol = max(m, n) * np.spacing(smax)
    sv = np.sqrt(np.maximum(d, 0.0))
    doubt = sv < 1e4 * np.sqrt(np.finfo(float).eps) * smax
    if doubt.any():
        sv[doubt] = np.linalg.norm(Js @ V[:, doubt], axis=0)
    rank = int(np.count_nonzero(sv > tol))
    W = NS(rank=rank, deficiency=n - rank)
    if W.deficiency > 0:
        k = np.argsort(np.abs(d), kind='stable')[:W.deficiency]      # :405-407
        W.V, W.d = V[:, k], d[k]
        W.trace = float(np.trace(G) + np.sqrt(np.finfo(float).eps) * n)
        pt = np.asarray(paramTypes, dtype=object)
        avg = np.sqrt(1.0 / n)
        W.suspectedParams = []
        for j in range(W.deficiency):                                # :412-422
            o = np.argsort(-np.abs(W.V[:, j]), kind='stable')
            v = W.V[o, j]
            keep = np.abs(v) > 0.5 * (avg + abs(v[0]))
            W.suspectedParams.append(NS(values=v[keep], indices=o[keep], params=list(pt[o[keep]])))
    return W


def _blockdiag(blocks):
    """(N,k,k) blocks → sparse (N*k)x(N*k) block-diagonal CSC matrix."""
    N, k, _ = blocks.shape
    base = np.repeat(np.arange(N) * k, k * k)
    rr = base + np.tile(np.repeat(np.arange(k), k), N)
    cc = base + np.tile(np.tile(np.arange(k), k), N)
    return sp.csc_matrix((blocks.reshape(-1), (rr, cc)), shape=(N * k, N * k))


def bundle_cov(s, e, *varargin):
    """bundle_cov.m:1-55: posterior covariances CIO/CEO/COP (block-diagonal, sparse), CIOF/CEOF/COPF
    (full) and CXX (all unknowns, x order), from the undamped factorisation on the device, times
    s0^2.  CXX and COPF are dense on the device and refused above 2 GB."""
    P = e.problem
    out = []
    for w in varargin:
        lw = w.lower()
        if lw == 'prepare':                               # factorisation lives on the device
            out.append(e)
        elif lw in ('cio', 'ceo', 'cop'):
            out.append(_blockdiag(P.cov(lw, e.s0)))
        elif lw == 'ciof' and np.all(np.asarray(s.IO.struct.block) == np.asarray(s.IO.struct.block)[:, :1]):
            # one shared camera (all the device path supports): every image carries the same NC x NC block
            # (bundle_cov.m:148-160 with deserial fanning one x element out to all images), so the full matrix
            # is that block tiled - no need for the dense camera-system inverse
            nImg = s.IO.val.shape[1]
            out.append(sp.csc_matrix(np.tile(P.cov('cio', e.s0)[0], (nImg, nImg))))
        elif lw in ('ciof', 'ceof'):
            Cc = P.cov('cxx_cam', e.s0)
            key = lw[1:3].upper()
            des = getattr(s.bundle.deserial, key)
            shape = getattr(s.bundle.est, key).shape
            N = shape[0] * shape[1]
            Cf = np.zeros((N, N))
            Cf[np.ix_(des.dest, des.dest)] = Cc[np.ix_(des.src, des.src)]   # bundle_cov.m:148-196
            out.append(sp.csc_matrix(Cf))
        elif lw == 'copf':
            Cop = P.cov('cxx_op', e.s0)                    # OP x OP block of CXX, x order
            des = s.bundle.deserial.OP
            N = 3 * s.OP.val.shape[1]
            nC = P.n - Cop.shape[0]
            Cf = np.zeros((N, N))
            Cf[np.ix_(des.dest, des.dest)] = Cop[np.ix_(des.src - nC, des.src - nC)]   # bundle_cov.m:148-196
            out.append(sp.csc_matrix(Cf))
        elif lw == 'cxx':
            out.append(P.cov('cxx', e.s0))                 # bundle_cov.m:138-145
        else:
            raise ValueError("bundle_cov: unknown covariance '%s'" % w)
    return out[0] if len(out) == 1 else out
