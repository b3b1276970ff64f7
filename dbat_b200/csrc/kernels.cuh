// kernels.cuh — device-side problem view and kernel declarations shared by the .cu files.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>
#include "model.cuh"
#include "tilechol.h"

#define DBAT_GW 24                 // Gram width: NSLOT(14) IO | 6 EO | 1 r | pad  (3 tiles of 8)
#define DBAT_GT 3                  // 8-wide tiles
#define DBAT_GTP 6                 // lower-triangular tile pairs
#define DBAT_GSZ (DBAT_GTP * 64)   // doubles per Gram in C-fragment tile layout
#define DBAT_COL_EO DBAT_NSLOT     // first EO column in the Gram
#define DBAT_COL_R (DBAT_NSLOT + 6)
#define DBAT_PSB 128                // observations per block of the point-side assembly kernel
#define DBAT_CHUNK 1024            // max observations per camera-side chunk (one CTA)
#define DBAT_PT_STRIDE 52          // doubles per point record: V[6] g[3] pad Wsh[14][3]
#define DBAT_PT_WSH 10
#define DBAT_W_STRIDE 18           // doubles per observation cross block W_o (6 EO x 3 OP)
#define DBAT_NCAM (DBAT_NSLOT + 6)  // camera-side parameters of one image: IO slots then EO
#define DBAT_WF_STRIDE (3 * DBAT_NCAM)

static_assert(DBAT_NSLOT + 7 <= DBAT_GW, "Gram width");

struct Chunk { int img, start, count, pad; };

// window Schur (schur_win.cu): header of one group of <= WIN_GP neighbouring points whose image lists have a
// union of <= DBAT_GRP_MAXM images.  A cluster is a run of consecutive groups whose unions together span
// <= WIN_MAXW images (the "window").
#define WIN_GP 14                  // points per group (K = 3 * 14 = 42 columns of the contraction)
#define WIN_MAXW 20                // images per window = largest ray count the grouped path takes
struct __align__(16) WinHdr {
    int m, ng, p0, pad;                         // images in the union, points, position of the first point in grp_pt
    int j[WIN_GP];                              // point ids
    int ob[WIN_GP];                             // first point-major observation of every point
    unsigned char wslot[WIN_MAXW];              // window slot of every image of the union (ascending)
    unsigned char obsOf[WIN_GP][WIN_MAXW];      // observation (offset inside the point) of point x union image; 255 = not seen
    unsigned char pad2[4];
};
static_assert(sizeof(WinHdr) == 432, "WinHdr layout");

// Device view of one problem (all pointers are device pointers).
struct DevProblem {
    int nImg, nOP, nObs, nK, nP, model;
    int n;                 // unknowns
    int nC;                // camera-side unknowns (IO+EO) = order of the reduced system
    int nChunks;
    int ldS;               // order of the padded reduced system (multiple of 64; the last row carries the rhs)
    int nPrior;
    // observations, camera-major (reference row order: obs k -> rows 2k,2k+1)
    const double2* uv_cm; const double2* isig_cm; const int* pt_cm; const int* img_cm;
    // observations, point-major
    const double2* uv_pm; const double2* isig_pm; const int* img_pm; const int* pm2cm;
    const int* pt_start;   // nOP+1
    // point-side assembly: blocks of whole points with at most DBAT_PSB observations (one thread per observation);
    // points with more observations than that go through the one-thread-per-point kernel
    const int* psb_pt;     // nPsb pairs [first point, end point) of every block
    int nPsb;
    const int* psbig;      // points with more than DBAT_PSB observations
    int nPsbig;
    const Chunk* chunks;
    // current parameter values
    double* IOval; double* EOval; double* OPval;   // NC x nImg, 6 x nImg, 3 x nOP
    ImgRec* img; IORec* io;
    const int* img_io;     // nImg: index of every image's IO record (the io field of ImgRec, for the staging copy)
    // column maps (0-based x column, -1 = fixed)
    const int* sh_col;     // NSLOT
    const int* eo_col;     // nImg x 6
    const int* op_col;     // nOP x 3
    // position of the camera-side unknowns in the reduced system ("S order": images in elimination
    // order, shared IO last; tilesym.cu), -1 = fixed
    const int* sh_s;       // NSLOT
    const int* eo_s;       // nImg x 6
    const int* s2x;        // ldS: x column of every S index (-1: padding / rhs row)
    // general IO block structure (image-variant parameters, several cameras: IO.struct.block, buildserialindices.m:162-221)
    int ioGeneral;         // 0: one IO block shared by all images (fast path); 1: per-image column maps below are used
    int evalCompact;       // 1: every estimated IO slot is one of f, pp, b1, K1-K3, P1-P2 (nK <= 3, nP <= 2): compact evaluation kernels
    const int* cam_colx;   // nImg x 20: x column of [NSLOT IO slots | 6 EO elements] of every image (-1 fixed); both modes
    const int* cam_s;      // nImg x 20: the same as S indices
    double* Wfull;         // general mode: nObs x 60, cross blocks [IO slots | EO] x OP of every observation (point-major)
    int nGlob;             // IO columns used by more than one image (they sit last in S)
    const int* glob_x;     // nGlob: their x columns
    TCholDev T;            // the reduced system itself: 64 x 64 tiles of the sparse pattern (tilechol.cu)
    // prior observations
    const int* prior_col; const double* prior_val; const double* prior_isig;
    // normal-equation storage
    double* chunkG;        // nChunks x GSZ   partial Grams
    double* imgG;          // nImg x GSZ      per-image Gram (IO|EO|r)
    double* shG;           // GSZ             sum over images
    double* pt;            // nOP x PT_STRIDE point records
    double* W;             // nObs x 18       cross blocks, point-major order
    double* rhs;           // ldS             reduced right-hand side (S order)
    const int* pt_pm;      // point of every point-major observation
    // Schur reduction: estimated points sorted by their image list; a group is a run of <= WIN_GP neighbouring
    // points whose image lists have a union of at most 12 images (schur_win.cu)
    const int* grp_pt;     // point ids, grouped
    int grpMaxRays;        // largest union among the groups (sizes the window kernel's operand)
    const int* big_pt;     // the wide points: estimated points with more than DBAT_GRP_MAXM rays, ascending id
    int nBig;
    // wide-point Schur (schur_wide.cu): their observations numbered point by point ("wide observations"), the per-image
    // lists of them, the camera-pair blocks they touch and the staged factors Z_o = M_j W_o', [Wsh_j g_j]' M_j'
    const int* wide_o;     // nWObs: point-major observation of every wide observation
    const int* wimg_ptr;   // nImg+1: wide observations of every image ...
    const int* wimg_w;     // ... their numbers, ascending point
    const int* wimg_pt;    // ... their wide points (index into big_pt)
    const int* wpair;      // nWPair x (image A, image B), rank A >= rank B
    int nWObs, nWPair;
    double* wide_Z;        // nWObs x 18: Z_o[k][a], k = point coordinate, a = EO element
    double* wide_Zsh;      // nBig x 48: [k][s], s = shared IO slot 0..13, 14 = gradient, 15 = zero
    double* wide_ssPart;   // per DBAT_WIDE_SSPART wide points: their 16 x 16 shared x shared table
    double* wide_shAcc;    // NSLOT x (NSLOT+1): the sum of the partial tables (k_schur_ss_apply's shAcc)
    double* vinv;          // nOP x 8: (V_j + lambda I)^-1 (6 entries) for dbat_cov (launch_point_vinv)
    // window Schur (schur_win.cu): clusters of consecutive groups accumulate their camera x camera blocks in
    // shared memory; every cluster leaves ONE image of its window in a staging buffer and a second kernel sums the
    // images per block of S in a fixed order (index built at create) - no atomics, bit-reproducible
    const WinHdr* win_hdr; // one per group
    const int* clu_grp;    // nClu+1: first group of every cluster
    const int* clu_order;  // nClu: cluster ids, most groups first (launch order)
    const int* clu_img_off;      // nClu+1 offsets into clu_img
    const int* clu_img;    // window images of every cluster (ascending elimination rank)
    const long long* clu_stg;    // nClu+1 offsets (doubles) of the cluster images in win_stg
    int nClu, nCand;
    double* winM;          // nCand x 6: inv(chol(V_j + lambda I)) of the grouped points, in grp_pt order
    double* win_stg;       // staging: per cluster [window blocks (lower, 36 each) | 16 x 6*WIN_MAXW shared rows | 16 x 16]
    const int* red_ptr;    // nRedBlk+1: contributions of every camera-pair block of S
    const int* red_imgA; const int* red_imgB;   // images of the block (rank A >= rank B)
    const long long* red_off;    // staging offset of every contribution (36 doubles)
    int nRedBlk;
    const int* redi_ptr;   // nImg+1: contributions to the shared-IO x EO rows of every image
    const long long* redi_off;   // staging offset of entry (shared row 0, EO element 0) of the contribution
    double* win_ssPart;    // per 256 clusters: partial sums of the 16 x 16 shared x shared tables
};
#define DBAT_GRP_MAXM 20   // grouped path up to 20 rays per point (= WIN_MAXW); more rays: schur_wide.cu
#define DBAT_WIDE_SSPART 16   // wide points per partial shared x shared table
