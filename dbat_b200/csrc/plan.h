// plan.h — host-side plan of a problem: everything dbat_create (api.cu) derives from a dbat_problem_desc before it
// uploads anything.  The column maps, the observation orders, the co-visibility graph, the point-side assembly
// blocks and the window Schur index are built here from the description and the symbolic analysis alone, so
// none of it needs a device.
#pragma once
#include <string>
#include <vector>

#include "../../include/dbat_gpu.h"
#include "kernels.cuh"
#include "tilesym.h"

// What the handle keeps on the host for the life of the problem: Jacobian export, rank tests, covariance layout
// and the re-tiling for several ranks or devices.
struct ProblemPlan {
    int nImg = 0, nOP = 0, nObs = 0;
    int n = 0;                    // unknowns
    int NC = 0;                   // IO parameters per image: 5 + nK + nP
    int nC = 0;                   // camera-side unknowns x[0:nC]
    int m = 0;                    // residuals: two per observation, one per prior observation
    int nIOrec = 0;               // distinct IO records
    bool legacy = false;          // distModel 1 / -1
    bool general = false;         // not one IO block shared by all images (IO.struct.block, multi_res.m:92-111)
    int grpMaxPts = 0;            // most points in one window Schur group (dbat_reduced_info)
    // column maps (0-based x column, -1 = fixed)
    std::vector<int> io_col;      // NC x nImg
    std::vector<int> eo_col;      // 6 x nImg
    std::vector<int> op_col;      // 3 x nOP
    std::vector<int> io_colx;     // nImg x NSLOT: x column of every (image, IO slot)
    std::vector<int> sh_col;      // NSLOT: the shared column of every IO slot (all -1 with general IO)
    std::vector<int> glob_x;      // IO columns used by more than one image (all of them with one shared block)
    std::vector<int> colLocalImg; // per camera-side x column: the one image that uses this IO column, or -1
    std::vector<int> x2s;         // x column (camera side) -> S index
    // observations: k = camera-major (the description's order), o = point-major
    std::vector<int> img_cm, pt_cm;   // nObs
    std::vector<int> img_start;       // nImg + 1: observations k of every image
    std::vector<int> pt_start;        // nOP + 1: observations o of every point
    std::vector<int> pm2cm;           // nObs: k of every o
    // prior observations
    std::vector<int> prior_col;
    std::vector<double> prior_isig;
    // reduced system: co-visibility graph (CSR) and the columns every image has in S (EO elements and the IO
    // columns only it uses)
    std::vector<int64_t> adjPtr;
    std::vector<int32_t> adj;
    std::vector<int> nEO;
};

// Arrays that only exist to be uploaded; dbat_create drops them once they are on the device.
struct PlanUpload {
    // observations and camera-side records
    std::vector<double2> uv_cm, isig_cm, uv_pm, isig_pm;
    std::vector<int> img_pm, pt_pm;   // image / point of every point-major observation
    std::vector<Chunk> chunks;
    std::vector<int> img_chunk_start; // nImg + 1
    std::vector<int> ioOfImg, rep;    // IO record of every image, first image of every IO record
    std::vector<ImgRec> recs;
    std::vector<double> prior_val;
    std::vector<int> col2pt;          // point-side x column - nC -> 3 * point + coordinate
    // point-side assembly blocks
    std::vector<int> psb_pt, psbig;
    int nPsb = 0, nPsbig = 0;
    // window Schur index
    std::vector<int> grp_pt, big_pt;
    int nCand = 0, nBig = 0, grpMaxRays = 1;
    std::vector<WinHdr> win_hdr;
    std::vector<int> clu_grp, clu_order, clu_img_off, clu_img;
    std::vector<long long> clu_stg;
    std::vector<int> red_ptr, red_imgA, red_imgB, redi_ptr;
    std::vector<long long> red_off, redi_off;
    int nClu = 0, nRedBlk = 0;
};

// S index maps of the camera-side columns for one tiling of the reduced system
struct ReducedMaps {
    std::vector<int> sh_s, eo_s, s2x, cam_colx, cam_s;
};

// Stages in the order dbat_create runs them.  A stage that checks the description returns a DBAT_* code and
// sets err; the checks run in a fixed order, so the first failing one names the problem.
// The deserialisation maps, nC, the observation list (which images are observed decides shared vs general IO),
// the legacy expansion and the IO / EO structure checks.
int plan_columns(const dbat_problem_desc* d, ProblemPlan& p, std::string& err);
// unique IO records, image records, weights, the point-major order, camera-side chunks
void plan_observations(const dbat_problem_desc* d, ProblemPlan& p, PlanUpload& u);
// prior observations, m, col2pt
int plan_priors(const dbat_problem_desc* d, ProblemPlan& p, PlanUpload& u, std::string& err);
// co-visibility graph (with the description's covis edges), S columns per image, global IO
int plan_cameras(const dbat_problem_desc* d, ProblemPlan& p, const PlanUpload& u, std::string& err);
// runs of whole points for the point-side assembly and the list of long points
void plan_point_blocks(const ProblemPlan& p, PlanUpload& u);
// window Schur index for the elimination order of sym: groups, clusters, headers, reduction CSR, cluster order;
// estimated points with more than grpMaxM rays go to k_schur_atomic instead
void plan_schur_windows(ProblemPlan& p, PlanUpload& u, const TileSym& sym, int grpMaxM);
// sets p.x2s and returns the other S index maps
ReducedMaps plan_reduced_maps(ProblemPlan& p, const TileSym& sym);

// true when the images with columns in S come in the same elimination order in a and b
bool plan_same_order(const ProblemPlan& p, const TileSym& a, const TileSym& b);
// the compact evaluation kernels (eval.cu) apply
bool plan_eval_compact(const ProblemPlan& p, int nK, int nP);
// doubles of the block-partials buffer of the reductions
int plan_partials(const ProblemPlan& p, const PlanUpload& u);
