/* dbat_gpu.h — C ABI of libdbatgpu.so, the B200-native bundle-adjustment inner loop.
 *
 * Drop-in boundary for the hot path of niclasborlin/dbat (reference paths below are
 * relative to the reference checkout).  The reference has no FFI for this path; the
 * only precedent is its experimental MEX set (code/test/postcov/icpc_mex.c:495-611:
 * gateway validates inputs, MATLAB owns every returned array, errors are raised as
 * "DBAT:<fn>:<id>").  This ABI is what a MEX gateway (mex/dbat_mex.c) or the ctypes
 * host layer (dbat_b200/_lib.py) binds.  Plain pointers and sizes only; the library
 * copies every input (caller keeps ownership) and writes results into caller-allocated
 * buffers.  Index vectors are 1-based int64 exactly as MATLAB holds them.
 *
 * Entry point                         replaces (reference file:line)
 *   dbat_create / dbat_destroy         resFun=@(x)brown_euler_cam4(x,s) closure + W
 *                                      (code/bundle/bundle.m:156-175)
 *   dbat_eval                          [f,J]=brown_euler_cam4(x,s)
 *                                      (code/bundle/cameramodel/brown_euler_cam4.m:22-183,
 *                                       multi_res.m:14-315, lsa/prior_obs.m:28-65)
 *   dbat_jacobian_nnz/_csc             sparse J returned by the same call (multi_res.m:313)
 *   dbat_solve (method LM)             code/bundle/lsa/levenberg_marquardt.m:54-247
 *   dbat_solve (method LMP)            code/bundle/lsa/levenberg_marquardt_powell.m:60-335
 *   dbat_solve (method GNA)            code/bundle/lsa/gauss_newton_armijo.m:75-290
 *   dbat_cov                           code/bundle/bundle_cov.m:63-478
 *   dbat_comm_init                     (new) NCCL communicator for point-sharded runs
 *
 * Not thread-safe per handle.  All functions return 0 or a negative DBAT_E_* code and
 * never throw; dbat_last_error() gives the message.  Optimiser OUTCOME codes keep the
 * reference's values (0 ok, -1 max iterations, -2 singular, -3 line search, -4
 * structural rank) in dbat_result.code.
 */
#ifndef DBAT_GPU_H
#define DBAT_GPU_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DBAT_OK             0
#define DBAT_E_BADARG      -101
#define DBAT_E_CUDA        -102
#define DBAT_E_NCCL        -103
#define DBAT_E_OOM         -104
#define DBAT_E_NOTSPD      -105
#define DBAT_E_UNSUPPORTED -106
#define DBAT_E_STATE       -107

#define DBAT_METHOD_GM  0
#define DBAT_METHOD_GNA 1
#define DBAT_METHOD_LM  2
#define DBAT_METHOD_LMP 3

/* which-selectors of dbat_cov (bundle_cov.m:135-214) */
#define DBAT_COV_CIO  1   /* out: NC x NC x nImg  (zero rows/cols for fixed elements) */
#define DBAT_COV_CEO  2   /* out: 6 x 6 x nImg */
#define DBAT_COV_COP  3   /* out: 3 x 3 x nOP */
#define DBAT_COV_CXX_CAM 4 /* out: nCam x nCam dense covariance of the IO+EO unknowns (x order) */
#define DBAT_COV_CXX  5   /* out: n x n dense covariance of all unknowns, x order (bundle_cov.m:138-145);
                             refused with DBAT_E_UNSUPPORTED when the dense result would exceed 2 GB */
#define DBAT_COV_CXX_OP 6 /* out: (n - nCam) x (n - nCam): the OP x OP block of CXX (source of COPF) */

typedef struct dbat_handle dbat_handle;

/* Flat view of the DBAT struct `s` (code/misc/emptydbatstruct.m:8-182) after
 * buildserialindices (code/misc/buildserialindices.m:57-221).  Matrices are
 * column-major double as MATLAB stores them. */
typedef struct dbat_problem_desc {
    int64_t nImg, nOP, nIP;       /* images, object points, image points                */
    int32_t distModel, nK, nP;    /* s.IO.model.*  (NC = 5+nK+nP rows in IOval)          */
    const double  *IOval;         /* NC x nImg   s.IO.val [cc;px;py;as;sk;K..;P..]       */
    const double  *EOval;         /* 6  x nImg   s.EO.val [X;Y;Z;omega;phi;kappa]        */
    const double  *OPval;         /* 3  x nOP    s.OP.val                                */
    const double  *IPval;         /* 2  x nIP    s.IP.val (pixels), columns sorted by (image, OP) */
    const double  *IPstd;         /* 2  x nIP    s.IP.std (pixels)                       */
    const int64_t *IPimg;         /* nIP  image (1-based) of every IP column: [~,j]=find(s.IP.vis) */
    const int64_t *IPop;          /* nIP  OP column (1-based): [i,~]=find(s.IP.vis)      */
    const double  *pxSize;        /* 2  x nImg   s.IO.sensor.pxSize                      */
    int64_t n;                    /* s.bundle.serial.n, number of unknowns               */
    const int64_t *IOdes_src, *IOdes_dest; int64_t nIOdes;  /* s.bundle.deserial.IO      */
    const int64_t *EOdes_src, *EOdes_dest; int64_t nEOdes;  /* s.bundle.deserial.EO      */
    const int64_t *OPdes_src, *OPdes_dest; int64_t nOPdes;  /* s.bundle.deserial.OP      */
    /* prior observations in residual-row order IO,EO,OP (prior_obs.m:28-65):
     * x index = serial.*.dest(serial.*.obs), value = prior.*.val(src(obs)),
     * std = prior.*.std(use) */
    int64_t nPriorIO, nPriorEO, nPriorOP;
    const int64_t *prior_x;       /* nPriorIO+nPriorEO+nPriorOP, 1-based                 */
    const double  *prior_val, *prior_std;
    /* Optional: co-visibility edges (pairs of 1-based image indices that observe a common object point) of
     * the WHOLE project.  A point-sharded problem (one rank of a multi-GPU run) sees only its own points, but
     * every rank must order and tile the reduced camera system identically; nCovis == 0: use the local points. */
    int64_t nCovis;
    const int64_t *covis_a, *covis_b;
} dbat_problem_desc;

/* Optimiser constants; defaults are those hard-coded in bundle.m:281-283,301-304,321-325. */
typedef struct dbat_opts {
    int32_t maxIter;        /* bundle.m:78 (20) */
    double  convTol;        /* bundle.m:87 (1e-6) */
    int32_t absTerm;        /* bundle.m:186-192 */
    int32_t singularTest;   /* GNA only */
    int32_t doTrace;        /* print one line per iteration */
    double  lambda0, lambdaMin;  /* LM: negative => scaled by trace(J0'J0)/n (-1e-10) */
    double  delta0;              /* LMP: <=0 => norm(x0) */
    double  mu, eta;             /* GNA: mu=0.1 ; LMP: mu=rhoBad 0.25, eta=rhoGood 0.75 */
    double  alphaMin;            /* GNA 1e-9 */
} dbat_opts;

/* Caller-allocated result buffers (MATLAB-owned in the MEX gateway). cap = maxIter+2. */
typedef struct dbat_result {
    double  *x;             /* n        final estimate */
    double  *p;             /* n        final step (final.p) */
    double  *r_w, *r_u;     /* m        final weighted / unweighted residual (may be NULL) */
    double  *trace;         /* n x cap  iteration trace T (may be NULL) */
    double  *rr;            /* cap+1    residual norms */
    double  *damping;       /* cap+1    lambdas (LM) / deltas (LMP) / alphas (GNA) */
    double  *rhos;          /* cap      LMP gain ratios (may be NULL) */
    int32_t *steps;         /* cap      LMP step types (may be NULL) */
    int32_t  code;          /* 0, -1, -2, -3, -4 as in the reference */
    int32_t  iters;         /* n (trial count for LM) */
    int32_t  nTrace, nRr, nDamping, nRhos;   /* used lengths */
    double   seconds;       /* wall time inside the optimiser loop */
    int64_t  launches;      /* CUDA kernels launched by this call */
} dbat_result;

int  dbat_create(const dbat_problem_desc *desc, dbat_handle **out);
void dbat_destroy(dbat_handle *h);
const char *dbat_last_error(const dbat_handle *h);   /* h may be NULL: last create error */

int64_t dbat_num_unknowns(const dbat_handle *h);
int64_t dbat_num_residuals(const dbat_handle *h);

/* Residual (and Jacobian state) at x.  r (length m, may be NULL) receives the
 * UNWEIGHTED residual in reference row order; weighted!=0 gives R*f instead. */
int dbat_eval(dbat_handle *h, const double *x, double *r, int weighted);

/* Sparse Jacobian at the x of the last dbat_eval / dbat_solve, MATLAB CSC layout
 * (Jc n+1 column pointers 0-based, Ir 0-based rows, exact zeros dropped as
 * find()/sparse() do in multi_res.m:150-313). Call _nnz first, allocate, then _csc. */
int dbat_jacobian_nnz(dbat_handle *h, int weighted, int64_t *nnz);
int dbat_jacobian_csc(dbat_handle *h, int weighted, int64_t *Jc, int64_t *Ir, double *vals);

void dbat_default_opts(int method, dbat_opts *opts);
int  dbat_solve(dbat_handle *h, int method, const dbat_opts *opts, const double *x0,
                dbat_result *res);

/* One pass of the hot path at x without optimiser logic (bench + tests):
 * residual+Jacobian+assembly, Schur with damping lambda, Cholesky, back-substitution.
 * x == NULL reuses the device-resident iterate; p (n, may be NULL) receives the step.
 * flags: bit0 Jacobi column scaling, bit1 also evaluate the trial point x+p, bit2 accept the
 * trial point when f decreases (one Levenberg-Marquardt iteration).
 * stats (8 doubles): [0] f=1/2 r'r, [1] |Jp|^2, [2] r'Jp, [3] singular flag, [4] kernel
 * launches, [5] f(x+p) or NaN, [6] device time in ms (CUDA events on the library stream). */
int dbat_normal_step(dbat_handle *h, const double *x, double lambda, int flags,
                     double *p, double *stats);

/* Posterior covariances from the undamped factorisation at the current x, times s0^2. */
int dbat_cov(dbat_handle *h, int which, double s0, double *out);

/* Report-side consumers of the posterior covariance, computed on the device from ONE factorisation (SURVEY §8f N2).
 * Replaces the host post-processing of code/bundle/bundle_result_file.m:92-153 (standard deviations),
 * code/misc/corrmat.m:21-47 and code/bundle/private/high_{io,eo,op}_correlations.m (block form):
 *   std_x[n]  posterior standard deviation of every unknown, x order (NaN after a failed factorisation);
 *   io/eo/op  the pairs of one block whose correlation exceeds `thres` in magnitude - IO: the NC x NC block of
 *             every image (images of one camera hold identical blocks; rows in the struct's IO order), EO: 6 x 6 per
 *             image, OP: 3 x 3 per object point - in the reference's order (block, then column, then row).
 * A list may be NULL.  `n` returns the number of pairs found; at most `cap` are stored.  Indices are 0-based. */
typedef struct dbat_cov_hit_list {
    int64_t  cap;            /* in: capacity of the arrays */
    int64_t  n;              /* out: pairs found */
    int64_t *block;          /* image or object point of the pair */
    int32_t *row, *col;      /* positions inside the block, row > col */
    double  *rho;            /* correlation, clipped to [-1, 1] */
} dbat_cov_hit_list;
int dbat_cov_stats(dbat_handle *h, double s0, double thres, double *std_x, dbat_cov_hit_list *io,
                   dbat_cov_hit_list *eo, dbat_cov_hit_list *op);

/* Elimination order of the images for a banded factorisation of the reduced camera system (host only, no
 * device needed): reverse Cuthill-McKee on the co-visibility graph - images i, j are adjacent when they
 * observe a common object point, which is exactly when S has a non-zero 6x6 block (i, j).  obs_img / obs_op
 * are 1-based as in dbat_problem_desc; perm (nImg, 1-based) lists the images in elimination order and
 * *bandwidth (may be NULL) is the largest distance, in images, between two adjacent images under it.  The
 * reference has no counterpart on its solver path (it factors the camera block densely, bundle_cov.m:97);
 * its ordering experiments are private/blkcolperm.m and test/postcov/reorder_test.m. */
int dbat_camera_order(int64_t nImg, int64_t nOP, int64_t nObs, const int64_t *obs_img,
                      const int64_t *obs_op, int64_t *perm, int64_t *bandwidth);

/* Structure of the reduced camera system of a problem: info (16) = {nT (64 x 64 tile rows), ld, nS (camera-side
 * unknowns), nSlots (stored tiles incl. fill), nSlotsS (tiles of S itself), nTasks, nTerms (tile products per
 * factorisation), depth (longest dependency chain in tile columns), order mode, segments, grid of the factorisation,
 * grid of the backward solve, then which point-side paths the problem takes:
 *   [12] points with more than 128 observations (one-thread-per-point assembly and back-substitution, or one block
 *        per point in several passes with general IO),
 *   [13] estimated points with more than 20 observations (per-point Schur kernel with FP64 atomics),
 *   [14] largest union of image lists of one window Schur group (above 12 the wider window instantiation runs),
 *   [15] most points in one window Schur group}. */
int dbat_reduced_info(const dbat_handle *h, int64_t *info);

/* Symbolic analysis of the reduced camera system on its own (host only; tests and tools): elimination order
 * of the images (mode 0 natural, 1 reverse Cuthill-McKee, 2 nested dissection, -1 automatic), 64 x 64 tile
 * pattern with fill, task list of the data-flow factorisation.  nEO (nImg): estimated EO elements per image;
 * counts (16) = {nT, ld, nS, nSlots, nSlotsS, nTasks, nTerms, depth, mode, nSeg, ioS}.  dbat_tile_symbolic_get
 * copies the arrays of the last analysis (any pointer may be NULL): imgS (nImg), tix (nT*nT), taskIJ
 * (2*nTasks), termPtr (nTasks+1), termAB (2*nTerms), level (nT), s2kind (ld), bwdCols (nT). */
int dbat_tile_symbolic(int64_t nImg, int64_t nOP, int64_t nObs, const int64_t *obs_img, const int64_t *obs_op,
                       const int64_t *nEO, int64_t nIO, int64_t mode, int64_t leafImages, int64_t *counts);
int dbat_tile_symbolic_get(int64_t *imgS, int64_t *tix, int64_t *taskIJ, int64_t *termPtr, int64_t *termAB,
                           int64_t *level, int64_t *s2kind, int64_t *bwdCols);
/* Distributed factorisation: counts[14], counts[15] of dbat_tile_symbolic are, on entry, the number of parts the
 * elimination tree is cut into and the part whose task lists are wanted (0, 0: one part); on return counts[11..15] =
 * {nTasks1 (tasks of phase 1), nTopS, nTop (slots of the top tile columns), parts actually used, nOwnS}.
 * dbat_tile_symbolic_get2: taskMode (nTasks; 1 = partial sum), colOwner (nT; -1 = top), ownSBegin (parts + 1). */
int dbat_tile_symbolic_get2(int64_t *taskMode, int64_t *colOwner, int64_t *ownSBegin);
/* Station coordinates (3 x nImg) for the next dbat_tile_symbolic call: the dissection then bisects geometrically
 * (dbat_create takes them from EOval); nImg = 0 / NULL clears them. */
int dbat_tile_symbolic_coords(int64_t nImg, const double *xyz);

/* The sparse tile solver on its own (unit tests / profiling): x = A^-1 b for a symmetric positive definite
 * column-major n x n matrix whose 6-column blocks play the role of images (coupled where A has a non-zero),
 * through the ordering, symbolic analysis and data-flow tile Cholesky the reduced camera system uses.
 * mode as in dbat_tile_symbolic; stats (8, may be NULL) = {ms best of `repeat`, nT, nSlots, nTasks, nTerms,
 * depth, min pivot, max pivot}. */
int dbat_tile_chol_solve(int64_t n, const double *A, const double *b, double *x, int64_t mode, int64_t leafImages,
                         int repeat, double *stats);

/* The dense inverse on its own (unit tests / profiling): Ainv (n x n) = A^-1 for a symmetric
 * positive definite column-major n x n matrix, through the blocked FP64 Cholesky and explicit
 * inverse dbat_cov runs on the reduced camera system.  DBAT_E_NOTSPD if a pivot is not positive.
 * ms_out (may be NULL): best device time of `repeat` factor+inverse passes (CUDA events). */
int dbat_dense_chol_inverse(int64_t n, const double *A, double *Ainv, int repeat, double *ms_out);

/* One process, several devices (SURVEY §8b; a MEX gateway has one interpreter thread): after dbat_create and before
 * the first evaluation, turn the handle into the front of `ndev` sub-problems, one per listed CUDA device.  The object
 * points are cut into one range per device, the sub-problems are joined by NCCL, and every later call on the handle
 * (dbat_eval, dbat_normal_step, dbat_solve, dbat_cov blocks, dbat_phase_times) runs on all of them and merges the
 * results; x, p and residuals keep the single-device layout.  Not available on a multi-device handle: the Jacobian
 * export and the dense point covariances (CXX / CXX_OP).  ndev = 1 moves the problem to dev[0]. */
int dbat_set_devices(dbat_handle *h, const int *dev, int ndev);

/* Multi-GPU: one process per GPU.  unique_id = the 128 bytes of ncclGetUniqueId from
 * rank 0 (dbat_comm_unique_id), distributed by the host plumbing (torch.distributed). */
int dbat_comm_unique_id(void *id128);
int dbat_comm_init(dbat_handle *h, int nranks, int rank, const void *id128);

/* Per-phase device time (ms) of the last dbat_solve / dbat_normal_step, for bench.py:
 * names[i] is a static string; returns the number of phases written (<= cap). */
int dbat_phase_times(const dbat_handle *h, const char **names, double *ms, int64_t *count, int cap);

/* ---- start values (SURVEY.md §8f N1) ------------------------------------------------------------
 * Forward intersection of object points from known IO/EO.  Replaces
 * code/photogrammetry/forwintersect.m:19-46 (pm_multiforwintersect.m:15-51, pm_forwintersect3.m:11-73,
 * lens correction pm_multilenscorr1.m:36-69).  All arrays are host arrays in MATLAB layout
 * (column-major doubles, 1-based int64 indices).  Points seen in fewer than two images get NaN. */
typedef struct dbat_fwi_desc {
    int64_t nImg, nOP, nObs, NC, nK, nP;
    const double*  IO;        /* NC x nImg  [f; ppx; ppy; b1; b2; K(nK); P(nP)] (the struct's storage) */
    const double*  EO;        /* 6 x nImg   [X;Y;Z;omega;phi;kappa] */
    const double*  pxSize;    /* 2 x nImg   mm per pixel */
    const double*  IPval;     /* 2 x nObs   measured pixel coordinates */
    const int64_t* obs_img;   /* nObs, image of every observation (1-based) */
    const int64_t* obs_op;    /* nObs, object point (column of OP) of every observation (1-based) */
    const int64_t* pts;       /* nPts, object points to compute (1-based) */
    int64_t nPts;
} dbat_fwi_desc;
/* OP: 3 x nPts out; res: nPts out or NULL (pm_forwintersect3's norm(b-Ax)/n); kernel_ms: device time or NULL */
int dbat_forwintersect(const dbat_fwi_desc* desc, double* OP, double* res, double* kernel_ms);
const char* dbat_forwintersect_error(void);

/* Batched 3-point spatial resection with residual test, one problem per camera.  Replaces the
 * per-camera body of code/photogrammetry/resect.m:96-129 (pm_resect_3pt.m:38-147: Grunert's quartic,
 * absolute orientation per admissible root, mean reprojection residual over the test points, best
 * root; then EO = [euclidean(null(P)); derotmat3d(P(:,1:3))]).  The caller chooses the three points
 * (largesttriangle.m) and passes lens-corrected, normalised image coordinates (K\[x;y;1]). */
typedef struct dbat_resect_desc {
    int64_t nCam;
    const double*  X3;          /* 3 x 3 x nCam  object coordinates of the three points (columns) */
    const double*  x3;          /* 2 x 3 x nCam  their normalised image coordinates */
    const int64_t* test_start;  /* nCam+1, 0-based offsets of every camera's test points in XT / xT */
    const double*  XT;          /* 3 x nTest     object coordinates of the test points */
    const double*  xT;          /* 2 x nTest     normalised image coordinates of the test points */
    int32_t behind;             /* pm_resect_3pt's `behind` flag (resect.m passes true) */
} dbat_resect_desc;
/* EO: 6 x nCam out ([X;Y;Z;omega;phi;kappa], NaN when no admissible root); res: nCam out (best mean residual).
 * Errors are reported through dbat_forwintersect_error(). */
int dbat_resect3(const dbat_resect_desc* desc, double* EO, double* res);

#ifdef __cplusplus
}
#endif
#endif /* DBAT_GPU_H */
