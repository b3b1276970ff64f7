"""ctypes binding of libdbatgpu.so (include/dbat_gpu.h).

This is the same C ABI a MATLAB MEX gateway binds (mex/dbat_mex.c).  There is no CPU
fallback: if the library is missing or no CUDA device is present, calls raise.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('DBAT_LIB', os.path.join(_HERE, 'libdbatgpu.so'))   # DBAT_LIB: tuning builds

METHOD = {'gm': 0, 'gna': 1, 'lm': 2, 'lmp': 3}
E_NOTSPD = -105        # DBAT_E_NOTSPD (include/dbat_gpu.h)
COV = {'cio': 1, 'ceo': 2, 'cop': 3, 'cxx_cam': 4, 'cxx': 5, 'cxx_op': 6}

c_dp = C.POINTER(C.c_double)
c_ip = C.POINTER(C.c_int64)


class ProblemDesc(C.Structure):
    _fields_ = [
        ('nImg', C.c_int64), ('nOP', C.c_int64), ('nIP', C.c_int64),
        ('distModel', C.c_int32), ('nK', C.c_int32), ('nP', C.c_int32),
        ('IOval', c_dp), ('EOval', c_dp), ('OPval', c_dp), ('IPval', c_dp), ('IPstd', c_dp),
        ('IPimg', c_ip), ('IPop', c_ip), ('pxSize', c_dp),
        ('n', C.c_int64),
        ('IOdes_src', c_ip), ('IOdes_dest', c_ip), ('nIOdes', C.c_int64),
        ('EOdes_src', c_ip), ('EOdes_dest', c_ip), ('nEOdes', C.c_int64),
        ('OPdes_src', c_ip), ('OPdes_dest', c_ip), ('nOPdes', C.c_int64),
        ('nPriorIO', C.c_int64), ('nPriorEO', C.c_int64), ('nPriorOP', C.c_int64),
        ('prior_x', c_ip), ('prior_val', c_dp), ('prior_std', c_dp),
        ('nCovis', C.c_int64), ('covis_a', c_ip), ('covis_b', c_ip),
    ]


class Opts(C.Structure):
    _fields_ = [
        ('maxIter', C.c_int32), ('convTol', C.c_double), ('absTerm', C.c_int32),
        ('singularTest', C.c_int32), ('doTrace', C.c_int32),
        ('lambda0', C.c_double), ('lambdaMin', C.c_double), ('delta0', C.c_double),
        ('mu', C.c_double), ('eta', C.c_double), ('alphaMin', C.c_double),
    ]


class Result(C.Structure):
    _fields_ = [
        ('x', c_dp), ('p', c_dp), ('r_w', c_dp), ('r_u', c_dp), ('trace', c_dp),
        ('rr', c_dp), ('damping', c_dp), ('rhos', c_dp), ('steps', C.POINTER(C.c_int32)),
        ('code', C.c_int32), ('iters', C.c_int32),
        ('nTrace', C.c_int32), ('nRr', C.c_int32), ('nDamping', C.c_int32), ('nRhos', C.c_int32),
        ('seconds', C.c_double), ('launches', C.c_int64),
    ]


EXPORTS = ['dbat_create', 'dbat_destroy', 'dbat_last_error', 'dbat_num_unknowns',
           'dbat_num_residuals', 'dbat_eval', 'dbat_jacobian_nnz', 'dbat_jacobian_csc',
           'dbat_default_opts', 'dbat_solve', 'dbat_normal_step', 'dbat_cov', 'dbat_cov_stats',
           'dbat_comm_unique_id', 'dbat_comm_init', 'dbat_phase_times', 'dbat_dense_chol_inverse',
           'dbat_forwintersect', 'dbat_forwintersect_error', 'dbat_resect3', 'dbat_camera_order',
           'dbat_tile_symbolic', 'dbat_tile_symbolic_get', 'dbat_tile_symbolic_get2', 'dbat_tile_symbolic_coords',
           'dbat_tile_chol_solve',
           'dbat_reduced_info', 'dbat_set_devices']

_lib = None


class CovHitList(C.Structure):
    """dbat_cov_hit_list (include/dbat_gpu.h): pairs of one block whose correlation exceeds the threshold."""
    _fields_ = [('cap', C.c_int64), ('n', C.c_int64), ('block', C.POINTER(C.c_int64)),
                ('row', C.POINTER(C.c_int32)), ('col', C.POINTER(C.c_int32)), ('rho', C.POINTER(C.c_double))]


class FwiDesc(C.Structure):
    _fields_ = [
        ('nImg', C.c_int64), ('nOP', C.c_int64), ('nObs', C.c_int64), ('NC', C.c_int64), ('nK', C.c_int64), ('nP', C.c_int64),
        ('IO', c_dp), ('EO', c_dp), ('pxSize', c_dp), ('IPval', c_dp),
        ('obs_img', c_ip), ('obs_op', c_ip), ('pts', c_ip), ('nPts', C.c_int64),
    ]


class ResectDesc(C.Structure):
    _fields_ = [
        ('nCam', C.c_int64), ('X3', c_dp), ('x3', c_dp), ('test_start', c_ip), ('XT', c_dp), ('xT', c_dp),
        ('behind', C.c_int32),
    ]


def lib():
    """Load libdbatgpu.so (raises if it has not been built: no fallback path exists)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError('libdbatgpu.so not built: run `python -m dbat_b200.build` '
                           '(or __graft_entry__.build()); there is no CPU fallback')
    L = C.CDLL(LIB_PATH)
    vp = C.c_void_p
    L.dbat_create.argtypes = [C.POINTER(ProblemDesc), C.POINTER(vp)]
    L.dbat_create.restype = C.c_int
    L.dbat_destroy.argtypes = [vp]
    L.dbat_destroy.restype = None
    L.dbat_last_error.argtypes = [vp]
    L.dbat_last_error.restype = C.c_char_p
    L.dbat_num_unknowns.argtypes = [vp]
    L.dbat_num_unknowns.restype = C.c_int64
    L.dbat_num_residuals.argtypes = [vp]
    L.dbat_num_residuals.restype = C.c_int64
    L.dbat_eval.argtypes = [vp, c_dp, c_dp, C.c_int]
    L.dbat_eval.restype = C.c_int
    L.dbat_jacobian_nnz.argtypes = [vp, C.c_int, C.POINTER(C.c_int64)]
    L.dbat_jacobian_nnz.restype = C.c_int
    L.dbat_jacobian_csc.argtypes = [vp, C.c_int, c_ip, c_ip, c_dp]
    L.dbat_jacobian_csc.restype = C.c_int
    L.dbat_default_opts.argtypes = [C.c_int, C.POINTER(Opts)]
    L.dbat_default_opts.restype = None
    L.dbat_solve.argtypes = [vp, C.c_int, C.POINTER(Opts), c_dp, C.POINTER(Result)]
    L.dbat_solve.restype = C.c_int
    L.dbat_normal_step.argtypes = [vp, c_dp, C.c_double, C.c_int, c_dp, c_dp]
    L.dbat_normal_step.restype = C.c_int
    L.dbat_cov.argtypes = [vp, C.c_int, C.c_double, c_dp]
    L.dbat_cov.restype = C.c_int
    L.dbat_cov_stats.argtypes = [vp, C.c_double, C.c_double, c_dp, C.POINTER(CovHitList), C.POINTER(CovHitList), C.POINTER(CovHitList)]
    L.dbat_cov_stats.restype = C.c_int
    L.dbat_comm_unique_id.argtypes = [C.c_void_p]
    L.dbat_comm_unique_id.restype = C.c_int
    L.dbat_comm_init.argtypes = [vp, C.c_int, C.c_int, C.c_void_p]
    L.dbat_comm_init.restype = C.c_int
    L.dbat_phase_times.argtypes = [vp, C.POINTER(C.c_char_p), c_dp, c_ip, C.c_int]
    L.dbat_phase_times.restype = C.c_int
    L.dbat_dense_chol_inverse.argtypes = [C.c_int64, c_dp, c_dp, C.c_int, c_dp]
    L.dbat_dense_chol_inverse.restype = C.c_int
    L.dbat_forwintersect.argtypes = [C.POINTER(FwiDesc), c_dp, c_dp, c_dp]
    L.dbat_forwintersect.restype = C.c_int
    L.dbat_forwintersect_error.argtypes = []
    L.dbat_forwintersect_error.restype = C.c_char_p
    L.dbat_resect3.argtypes = [C.POINTER(ResectDesc), c_dp, c_dp]
    L.dbat_resect3.restype = C.c_int
    L.dbat_camera_order.argtypes = [C.c_int64, C.c_int64, C.c_int64, c_ip, c_ip, c_ip, C.POINTER(C.c_int64)]
    L.dbat_camera_order.restype = C.c_int
    L.dbat_set_devices.argtypes = [vp, C.POINTER(C.c_int), C.c_int]
    L.dbat_set_devices.restype = C.c_int
    L.dbat_reduced_info.argtypes = [vp, c_ip]
    L.dbat_reduced_info.restype = C.c_int
    L.dbat_tile_symbolic.argtypes = [C.c_int64, C.c_int64, C.c_int64, c_ip, c_ip, c_ip, C.c_int64, C.c_int64,
                                     C.c_int64, c_ip]
    L.dbat_tile_symbolic.restype = C.c_int
    L.dbat_tile_symbolic_get.argtypes = [c_ip] * 8
    L.dbat_tile_symbolic_get.restype = C.c_int
    L.dbat_tile_symbolic_coords.argtypes = [C.c_int64, c_dp]
    L.dbat_tile_symbolic_coords.restype = C.c_int
    L.dbat_tile_symbolic_get2.argtypes = [c_ip] * 3
    L.dbat_tile_symbolic_get2.restype = C.c_int
    L.dbat_tile_chol_solve.argtypes = [C.c_int64, c_dp, c_dp, c_dp, C.c_int64, C.c_int64, C.c_int, c_dp]
    L.dbat_tile_chol_solve.restype = C.c_int
    _lib = L
    return L


def dptr(a):
    return a.ctypes.data_as(c_dp) if a is not None else None


def iptr(a):
    return a.ctypes.data_as(c_ip) if a is not None else None


def f64(a):
    return np.ascontiguousarray(np.asarray(a, dtype=np.float64))


def i64(a):
    return np.ascontiguousarray(np.asarray(a, dtype=np.int64))


class DbatError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__('libdbatgpu error %d: %s' % (code, msg))
        self.code = code


def dense_chol_inverse(A, repeat=1):
    """A^-1 through the dense factor + inverse of dbat_cov on the device; returns (Ainv, ms), ms the best device time
    of `repeat` passes."""
    A = np.asfortranarray(np.asarray(A, dtype=np.float64))
    n = A.shape[0]
    Ainv = np.empty((n, n), order='F')
    ms = C.c_double()
    rc = lib().dbat_dense_chol_inverse(n, A.ctypes.data_as(c_dp), Ainv.ctypes.data_as(c_dp), repeat, C.byref(ms))
    if rc != 0:
        raise DbatError(rc, lib().dbat_last_error(None).decode())
    return Ainv, ms.value


def camera_order(img, op, nImg, nOP):
    """Reverse Cuthill-McKee order of the images on the co-visibility graph (host code in the library):
    returns (perm, bandwidth) with perm 0-based."""
    img1, op1 = i64(np.asarray(img) + 1), i64(np.asarray(op) + 1)
    perm = np.empty(nImg, dtype=np.int64)
    bw = C.c_int64()
    rc = lib().dbat_camera_order(nImg, nOP, len(img1), iptr(img1), iptr(op1), iptr(perm), C.byref(bw))
    if rc != 0:
        raise DbatError(rc, 'dbat_camera_order: bad argument')
    return perm - 1, int(bw.value)


def tile_symbolic(img, op, nImg, nOP, nEO, nIO, mode=-1, leaf=120, parts=1, part=0, xyz=None):
    """Symbolic analysis of the reduced camera system (host code in the library): dict of counts + arrays.
    parts / part: task lists of one part of a distributed factorisation."""
    img1, op1, ne = i64(np.asarray(img) + 1), i64(np.asarray(op) + 1), i64(nEO)
    cnt = np.zeros(16, dtype=np.int64)
    cnt[14], cnt[15] = parts, part
    if xyz is not None:
        c = np.ascontiguousarray(np.asarray(xyz, dtype=np.float64).T)      # 3 x nImg column-major = nImg x 3 C order
        lib().dbat_tile_symbolic_coords(nImg, dptr(c))
    else:
        lib().dbat_tile_symbolic_coords(0, None)
    rc = lib().dbat_tile_symbolic(nImg, nOP, len(img1), iptr(img1), iptr(op1), iptr(ne), nIO, mode, leaf, iptr(cnt))
    if rc != 0:
        raise DbatError(rc, 'dbat_tile_symbolic failed')
    names = ['nT', 'ld', 'nS', 'nSlots', 'nSlotsS', 'nTasks', 'nTerms', 'depth', 'mode', 'nSeg', 'ioS', 'nTasks1',
             'nTopS', 'nTop', 'nParts', 'nOwnS']
    out = {k: int(cnt[i]) for i, k in enumerate(names)}
    nT = out['nT']
    arr = dict(imgS=np.empty(nImg, np.int64), tix=np.empty(nT * nT, np.int64), taskIJ=np.empty(max(1, 2 * out['nTasks']), np.int64),
               termPtr=np.empty(out['nTasks'] + 1, np.int64), termAB=np.empty(max(1, 2 * out['nTerms']), np.int64),
               level=np.empty(nT, np.int64), s2kind=np.empty(out['ld'], np.int64), bwdCols=np.empty(nT, np.int64))
    lib().dbat_tile_symbolic_get(*[iptr(arr[k]) for k in ('imgS', 'tix', 'taskIJ', 'termPtr', 'termAB', 'level', 's2kind', 'bwdCols')])
    arr2 = dict(taskMode=np.empty(max(1, 4 * out['nTasks']), np.int64), colOwner=np.empty(nT, np.int64),
                ownSBegin=np.empty(out['nParts'] + 1, np.int64))
    lib().dbat_tile_symbolic_get2(*[iptr(arr2[k]) for k in ('taskMode', 'colOwner', 'ownSBegin')])
    out.update(arr)
    out.update(arr2)
    out['tix'] = out['tix'].reshape(nT, nT)
    out['taskIJ'] = out['taskIJ'][:2 * out['nTasks']].reshape(-1, 2)
    tm = out['taskMode'][:4 * out['nTasks']].reshape(-1, 4)
    out['taskMode'], out['taskWait'], out['taskSet'], out['taskInit'] = tm[:, 0].copy(), tm[:, 1].copy(), tm[:, 2].copy(), tm[:, 3].copy()
    out['termAB'] = out['termAB'][:2 * out['nTerms']].reshape(-1, 2)
    out['bwdCols'] = out['bwdCols'][out['bwdCols'] >= 0]
    return out


def tile_chol_solve(A, b, mode=-1, leaf=120, repeat=1):
    """x = A^-1 b through the sparse tile Cholesky on the device; returns (x, stats dict)."""
    A = np.asfortranarray(np.asarray(A, dtype=np.float64))
    n = A.shape[0]
    b = f64(b)
    x = np.empty(n)
    st = np.zeros(8)
    rc = lib().dbat_tile_chol_solve(n, A.ctypes.data_as(c_dp), dptr(b), dptr(x), mode, leaf, repeat, dptr(st))
    if rc not in (0, E_NOTSPD):
        raise DbatError(rc, lib().dbat_last_error(None).decode())
    names = ['ms', 'nT', 'nSlots', 'nTasks', 'nTerms', 'depth', 'min_pivot', 'max_pivot']
    d = {k: float(st[i]) for i, k in enumerate(names)}
    d['rc'] = rc
    return x, d
