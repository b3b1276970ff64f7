// api.cu — C ABI (include/dbat_gpu.h), problem flattening, and the host-side optimiser
// drivers.  Control flow of the optimisers is copied literally from the reference
// (code/bundle/lsa/levenberg_marquardt.m:54-247, levenberg_marquardt_powell.m:60-335,
// gauss_newton_armijo.m:75-290); all vector work stays on the device and only a handful of
// scalars cross to the host per trial step.
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <map>
#include <string>
#include <iterator>
#include <vector>
#include <condition_variable>
#include <functional>
#include <memory>
#include <mutex>
#include <thread>
#include <dlfcn.h>

#include "../../include/dbat_gpu.h"
#include "kernels.cuh"
#include "launch.h"
#include "plan.h"
#include "tilechol.h"

int64_t g_dbat_launches = 0;
static std::string g_create_err;

#define CK(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess) {                                                                   \
            h->err = std::string(#call) + ": " + cudaGetErrorString(e_);                           \
            return DBAT_E_CUDA;                                                                    \
        }                                                                                          \
    } while (0)

enum { SC_RR = 0, SC_JP2 = 1, SC_RJP = 2, SC_TRACE = 3, SC_A = 4, SC_B = 5, SC_C = 6, SC_PRR = 7, SC_JPP = 8 /* 8..11 */, SC_RRT = 12, SC_N = 16 };
enum { PH_EVAL = 0, PH_SCHUR, PH_CHOL, PH_SOLVE, PH_TRIAL, PH_JP, PH_TOTAL, PH_N };
static const char* kPhaseNames[PH_N] = {"eval_jac_assembly", "build_schur", "cholesky", "solve_backsub",
                                        "trial_residual", "jp_stats", "total"};

// --------------------------------------------------------------------------------------------
// NCCL through dlopen (torch ships libnccl.so.2; no link-time dependency)
// --------------------------------------------------------------------------------------------
typedef struct { char internal[128]; } nccl_uid;
struct NcclApi {
    void* lib = nullptr;
    int (*GetUniqueId)(nccl_uid*) = nullptr;
    int (*CommInitRank)(void**, int, nccl_uid, int) = nullptr;
    int (*AllReduce)(const void*, void*, size_t, int, int, void*, cudaStream_t) = nullptr;
    int (*Reduce)(const void*, void*, size_t, int, int, int, void*, cudaStream_t) = nullptr;
    int (*GroupStart)() = nullptr;
    int (*GroupEnd)() = nullptr;
    int (*CommDestroy)(void*) = nullptr;
    const char* (*GetErrorString)(int) = nullptr;
};
static NcclApi g_nccl;
static bool nccl_load() {
    if (g_nccl.lib) return true;
    const char* names[] = {"libnccl.so.2", "libnccl.so"};
    for (const char* nm : names) { g_nccl.lib = dlopen(nm, RTLD_NOW | RTLD_GLOBAL); if (g_nccl.lib) break; }
    if (!g_nccl.lib) return false;
    g_nccl.GetUniqueId = (int (*)(nccl_uid*))dlsym(g_nccl.lib, "ncclGetUniqueId");
    g_nccl.CommInitRank = (int (*)(void**, int, nccl_uid, int))dlsym(g_nccl.lib, "ncclCommInitRank");
    g_nccl.AllReduce = (int (*)(const void*, void*, size_t, int, int, void*, cudaStream_t))dlsym(g_nccl.lib, "ncclAllReduce");
    g_nccl.Reduce = (int (*)(const void*, void*, size_t, int, int, int, void*, cudaStream_t))dlsym(g_nccl.lib, "ncclReduce");
    g_nccl.GroupStart = (int (*)())dlsym(g_nccl.lib, "ncclGroupStart");
    g_nccl.GroupEnd = (int (*)())dlsym(g_nccl.lib, "ncclGroupEnd");
    g_nccl.CommDestroy = (int (*)(void*))dlsym(g_nccl.lib, "ncclCommDestroy");
    g_nccl.GetErrorString = (const char* (*)(int))dlsym(g_nccl.lib, "ncclGetErrorString");
    return g_nccl.GetUniqueId && g_nccl.CommInitRank && g_nccl.AllReduce && g_nccl.Reduce && g_nccl.GroupStart && g_nccl.GroupEnd;
}

// --------------------------------------------------------------------------------------------
struct dbat_handle {
    std::string err;
    cudaStream_t st = nullptr, st2 = nullptr;
    cudaEvent_t evFork = nullptr, evJoin = nullptr, evStep = nullptr;
    DevProblem P{};
    ProblemPlan plan;                   // host-side index of the problem (plan.cu)
    // device allocations
    std::vector<void*> allocs;
    int *d_IOsrc = nullptr, *d_IOdst = nullptr, *d_EOsrc = nullptr, *d_EOdst = nullptr, *d_OPsrc = nullptr, *d_OPdst = nullptr;
    int nIOdes = 0, nEOdes = 0, nOPdes = 0;
    int *d_rep = nullptr, *d_img_chunk_start = nullptr, *d_col2pt = nullptr;
    double* d_pack = nullptr;                 // packed lower triangle of S for the multi-rank allreduce
    double *d_tmpG = nullptr, *d_partial = nullptr, *d_scal = nullptr;
    double* h_scal = nullptr;           // pinned
    double* h_G = nullptr;              // pinned: summed Gram of the last evaluation
    unsigned long long* h_piv = nullptr;   // pinned: min / max pivot and the breakdown flag of the last factorisation
    double* solve_pout = nullptr;       // step vector of a solve_step whose host-side part (finish_solve) is still due
    double *d_x = nullptr, *d_t = nullptr, *d_p = nullptr, *d_pgn = nullptr, *d_g = nullptr, *d_pc = nullptr;
    double* d_pEO = nullptr;             // nImg x 6: EO part of the last camera-side step per image (0 = fixed element)
    double *d_camDiag = nullptr, *d_camG = nullptr, *d_diagN = nullptr, *d_dscale = nullptr;
    double *d_evalRed = nullptr, *d_prr = nullptr; size_t nEvalRed = 0;
    double *d_r = nullptr;              // m doubles (export)
    TChol tc;                           // sparse tile Cholesky of the reduced system (tilechol.cu)
    double* d_dS = nullptr;             // Jacobi scale per S index
    unsigned long long* d_stats = nullptr;   // pivot statistics exchanged between the ranks
    const double* jp_vec = nullptr;     // vector whose |Jp|^2, r'Jp came out of the last back-substitution (nullptr: none)
    double jp_cache[2] = {0, 0};
    bool params_valid = false;          // parameter arrays correspond to d_x
    bool normal_valid = false;          // Gram / point records correspond to d_x
    // comm
    void* comm = nullptr; int nranks = 1, rank = 0;
    // a deep copy of the problem description (dbat_set_devices re-creates the problem per device from it)
    struct DescCopy* dcopy = nullptr;
    struct DevGroup* group = nullptr;   // non-null: this handle fronts one sub-problem per device
    // CSC cache
    std::vector<int64_t> cscJc, cscIr; std::vector<double> cscV; int cscWeighted = -1;
    // phase timing
    std::vector<cudaEvent_t> ev; size_t evUsed = 0;
    struct Span { int ph; size_t a, b; };
    std::vector<Span> spans;
    double phase_ms[PH_N] = {0}; int64_t phase_cnt[PH_N] = {0};
};

template <typename T>
static int dev_alloc(dbat_handle* h, T** p, size_t count) {
    if (count == 0) count = 1;
    cudaError_t e = cudaMalloc((void**)p, sizeof(T) * count);
    if (e != cudaSuccess) { h->err = std::string("cudaMalloc: ") + cudaGetErrorString(e); return DBAT_E_OOM; }
    h->allocs.push_back(*p);
    return 0;
}
template <typename T, typename U>        // U: T or const T
static int dev_upload(dbat_handle* h, U** p, const std::vector<T>& v) {
    T* q = nullptr;
    int rc = dev_alloc(h, &q, v.size());
    *p = q;
    if (rc) return rc;
    if (!v.empty()) {
        cudaError_t e = cudaMemcpy(q, v.data(), sizeof(T) * v.size(), cudaMemcpyHostToDevice);
        if (e != cudaSuccess) { h->err = std::string("cudaMemcpy: ") + cudaGetErrorString(e); return DBAT_E_CUDA; }
    }
    return 0;
}

static size_t ph_begin(dbat_handle* h) {
    if (h->evUsed + 2 > h->ev.size()) return (size_t)-1;
    size_t a = h->evUsed++;
    cudaEventRecord(h->ev[a], h->st);
    return a;
}
static void ph_end(dbat_handle* h, int ph, size_t a) {
    if (a == (size_t)-1) return;
    size_t b = h->evUsed++;
    cudaEventRecord(h->ev[b], h->st);
    h->spans.push_back({ph, a, b});
}
static void ph_reset(dbat_handle* h) {
    h->evUsed = 0; h->spans.clear();
    for (int i = 0; i < PH_N; ++i) { h->phase_ms[i] = 0; h->phase_cnt[i] = 0; }
}
static void ph_collect(dbat_handle* h) {
    cudaStreamSynchronize(h->st);
    for (auto& s : h->spans) {
        float ms = 0;
        cudaEventElapsedTime(&ms, h->ev[s.a], h->ev[s.b]);
        h->phase_ms[s.ph] += ms; h->phase_cnt[s.ph]++;
    }
    h->spans.clear(); h->evUsed = 0;
}

// --------------------------------------------------------------------------------------------
// create
// --------------------------------------------------------------------------------------------
static int fail_create(dbat_handle* h, int code, const std::string& msg) {
    g_create_err = msg;
    if (h) dbat_destroy(h);
    return code;
}

struct DescCopy;
static int group_eval(dbat_handle* h, const double* x, double* r, int weighted);
static int group_normal_step(dbat_handle* h, const double* x, double lambda, int flags, double* p, double* stats);
static int group_solve(dbat_handle* h, int method, const dbat_opts* opts, const double* x0, dbat_result* res);
static int group_cov(dbat_handle* h, int which, double s0, double* out);
static const dbat_handle* group_first(const dbat_handle* h);
static DescCopy* copy_desc(const dbat_problem_desc* d, int NC);
static void free_desc(DescCopy* c);
static void group_destroy(dbat_handle* h);
static thread_local bool g_in_group_create = false;

// Symbolic analysis of the reduced system for nParts parts (tilesym.cu).  dbat_create analyses it for one part;
// dbat_comm_init again when the factorisation is distributed over the ranks.
static int analyse_reduced(dbat_handle* h, int nParts, int myPart, TileSym& sym) {
    const ProblemPlan& pl = h->plan;
    if (tile_symbolic(pl.nImg, pl.adjPtr.data(), pl.adj.data(), pl.nEO.data(), (int)pl.glob_x.size(), -1, 120, sym, nParts,
                      myPart, pl.xyz.data())) {
        h->err = "symbolic analysis of the reduced system failed"; return DBAT_E_STATE;
    }
    return 0;
}

// (Re)build everything that depends on the tiling of the reduced system: the S index maps, the tile storage and the
// S-ordered work vectors.
static int setup_reduced(dbat_handle* h, const TileSym& sym) {
    DevProblem& P = h->P;
    const ReducedMaps mp = plan_reduced_maps(h->plan, sym);
    if (h->tc.d.tiles) tchol_free(h->tc);
    if (tchol_alloc(h->tc, sym)) { h->err = "out of memory for the reduced system"; return DBAT_E_OOM; }
    int rc = 0;
    if ((rc = dev_upload(h, &P.sh_s, mp.sh_s)) || (rc = dev_upload(h, &P.eo_s, mp.eo_s)) || (rc = dev_upload(h, &P.s2x, mp.s2x)) ||
        (rc = dev_upload(h, &P.cam_colx, mp.cam_colx)) || (rc = dev_upload(h, &P.cam_s, mp.cam_s)) ||
        (rc = dev_upload(h, &P.glob_x, h->plan.glob_x))) return rc;
    P.T = h->tc.d; P.nGlob = (int)h->plan.glob_x.size(); P.ldS = sym.ld;
    if ((rc = dev_alloc(h, &h->d_dS, (size_t)sym.ld)) || (rc = dev_alloc(h, &P.rhs, (size_t)sym.ld)) ||
        (rc = dev_alloc(h, &h->d_pc, (size_t)sym.ld))) return rc;
    if (!h->d_stats && (rc = dev_alloc(h, &h->d_stats, (size_t)4))) return rc;
    return 0;
}

static std::vector<int> zero_based(const int64_t* p, int64_t cnt) {
    std::vector<int> v(cnt);
    for (int64_t k = 0; k < cnt; ++k) v[k] = (int)(p[k] - 1);
    return v;
}

extern "C" int dbat_create(const dbat_problem_desc* d, dbat_handle** out) {
    if (!d || !out) { g_create_err = "null argument"; return DBAT_E_BADARG; }
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail_create(nullptr, DBAT_E_CUDA, "no CUDA device available (libdbatgpu has no CPU fallback)");
    dbat_handle* h = new dbat_handle();
    PlanOpts opts{DBAT_GRP_MAXM, getenv("DBAT_EVAL_GENERIC") != nullptr};
    // DBAT_GRP_MAXM=k lowers the threshold (tests of the per-point path)
    if (const char* e = getenv("DBAT_GRP_MAXM")) opts.grpMaxM = std::max(1, std::min(DBAT_GRP_MAXM, atoi(e)));

    // ---- host side: the plan (plan.cu) and the symbolic analysis of the reduced system
    ProblemPlan& pl = h->plan;
    PlanUpload up;
    TileSym sym;
    std::string msg;
    int rc = plan_columns(d, pl, msg);
    if (!rc) { plan_observations(d, pl, up); rc = plan_priors(d, pl, up, msg); }
    if (!rc) rc = plan_cameras(d, pl, up, msg);
    if (rc) return fail_create(h, rc, msg);
    if ((rc = analyse_reduced(h, 1, 0, sym))) return fail_create(h, rc, h->err);
    plan_point_blocks(pl, up);
    plan_schur_windows(pl, up, sym, opts);

    // ---- device side
    DevProblem& P = h->P;
    // kernel MODEL: 0..3 = res_euler_brown_0..3 (distModel 2..5); legacy 1 == model 2 arithmetic; -1 = forward Brown
    P.nImg = pl.nImg; P.nOP = pl.nOP; P.nObs = pl.nObs; P.nK = d->nK; P.nP = d->nP;
    P.model = pl.legacy ? (d->distModel == 1 ? 0 : 4) : d->distModel - 2;
    P.n = pl.n; P.nC = pl.nC; P.nChunks = (int)up.chunks.size(); P.nPrior = (int)pl.prior_col.size();
    P.ioGeneral = pl.general ? 1 : 0;
    P.evalCompact = plan_eval_compact(pl, d->nK, d->nP, opts) ? 1 : 0;
    P.nPsb = up.nPsb; P.nPsbig = up.nPsbig;
    P.nCand = up.nCand; P.nBig = up.nBig; P.grpMaxRays = up.grpMaxRays; P.nClu = up.nClu; P.nRedBlk = up.nRedBlk;
    if (cudaStreamCreate(&h->st) != cudaSuccess || cudaStreamCreateWithFlags(&h->st2, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreateWithFlags(&h->evFork, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&h->evJoin, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&h->evStep, cudaEventDisableTiming) != cudaSuccess)
        return fail_create(h, DBAT_E_CUDA, "cudaStreamCreate failed");
#define UP(ptr, vec) if ((rc = dev_upload(h, &ptr, vec)) != 0) return fail_create(h, rc, h->err)
#define AL(ptr, cnt) if ((rc = dev_alloc(h, &ptr, (size_t)(cnt)))) return fail_create(h, rc, h->err)
    UP(P.uv_cm, up.uv_cm); UP(P.isig_cm, up.isig_cm); UP(P.uv_pm, up.uv_pm); UP(P.isig_pm, up.isig_pm);
    UP(P.pt_cm, pl.pt_cm); UP(P.img_cm, pl.img_cm); UP(P.img_pm, up.img_pm); UP(P.pm2cm, pl.pm2cm);
    UP(P.pt_start, pl.pt_start); UP(P.chunks, up.chunks);
    UP(P.sh_col, pl.sh_col); UP(P.eo_col, pl.eo_col); UP(P.op_col, pl.op_col);
    UP(P.prior_col, pl.prior_col); UP(P.prior_val, up.prior_val); UP(P.prior_isig, pl.prior_isig);
    {
        std::vector<double> io(d->IOval, d->IOval + (size_t)pl.NC * pl.nImg), eo(d->EOval, d->EOval + (size_t)6 * pl.nImg),
            op(d->OPval, d->OPval + (size_t)3 * pl.nOP);
        UP(P.IOval, io); UP(P.EOval, eo); UP(P.OPval, op);
    }
    UP(P.img, up.recs); UP(P.img_io, up.ioOfImg);
    AL(P.io, pl.nIOrec);
    UP(h->d_rep, up.rep);
    h->nIOdes = (int)d->nIOdes; h->nEOdes = (int)d->nEOdes; h->nOPdes = (int)d->nOPdes;
    UP(h->d_IOsrc, zero_based(d->IOdes_src, d->nIOdes)); UP(h->d_IOdst, zero_based(d->IOdes_dest, d->nIOdes));
    UP(h->d_EOsrc, zero_based(d->EOdes_src, d->nEOdes)); UP(h->d_EOdst, zero_based(d->EOdes_dest, d->nEOdes));
    UP(h->d_OPsrc, zero_based(d->OPdes_src, d->nOPdes)); UP(h->d_OPdst, zero_based(d->OPdes_dest, d->nOPdes));
    UP(h->d_img_chunk_start, up.img_chunk_start); UP(h->d_col2pt, up.col2pt);
    if ((rc = setup_reduced(h, sym))) return fail_create(h, rc, h->err);
    const int nImg = pl.nImg, nOP = pl.nOP, nObs = pl.nObs;
    AL(P.chunkG, (size_t)std::max(1, P.nChunks) * DBAT_GSZ);
    {   // per-image Grams, their sum, camera-side prior terms and the prior r'r in ONE buffer: a multi-rank
        // evaluation sums it with a single allreduce
        const size_t nCp = (size_t)std::max(1, pl.nC);
        h->nEvalRed = (size_t)nImg * DBAT_GSZ + DBAT_GSZ + 2 * nCp + 8;
        AL(h->d_evalRed, h->nEvalRed);
        P.imgG = h->d_evalRed;
        P.shG = P.imgG + (size_t)nImg * DBAT_GSZ;
        h->d_camDiag = P.shG + DBAT_GSZ;
        h->d_camG = h->d_camDiag + nCp;
        h->d_prr = h->d_camG + nCp;
        // without prior observations the prior terms stay zero for the life of the handle (launch_prior_apply /
        // launch_prior_rr then queue nothing)
        cudaMemset(h->d_camDiag, 0, sizeof(double) * (2 * nCp + 8));
    }
    AL(P.pt, (size_t)std::max(1, nOP) * DBAT_PT_STRIDE);
    cudaMemset(P.pt, 0, sizeof(double) * (size_t)std::max(1, nOP) * DBAT_PT_STRIDE);   // the compact assembly leaves the rows of unestimated IO slots alone
    AL(P.W, (size_t)std::max(1, nObs) * DBAT_W_STRIDE);
    if (P.ioGeneral) AL(P.Wfull, (size_t)std::max(1, nObs) * DBAT_WF_STRIDE);
    UP(P.pt_pm, up.pt_pm);
    UP(P.psb_pt, up.psb_pt); UP(P.psbig, up.psbig);
    UP(P.grp_pt, up.grp_pt); UP(P.big_pt, up.big_pt);
    AL(P.vinv, (size_t)std::max(1, nOP) * 8);
    UP(P.clu_order, up.clu_order);
    UP(P.win_hdr, up.win_hdr); UP(P.clu_grp, up.clu_grp); UP(P.clu_img_off, up.clu_img_off); UP(P.clu_img, up.clu_img);
    UP(P.clu_stg, up.clu_stg); UP(P.red_ptr, up.red_ptr); UP(P.red_imgA, up.red_imgA); UP(P.red_imgB, up.red_imgB);
    UP(P.red_off, up.red_off); UP(P.redi_ptr, up.redi_ptr); UP(P.redi_off, up.redi_off);
    AL(P.winM, ((size_t)P.nCand + WIN_GP) * 6);
    AL(P.win_stg, (size_t)std::max<long long>(2, up.clu_stg.back()));
    AL(P.win_ssPart, (size_t)((P.nClu + 255) / 256 + 1) * 256);
    AL(h->d_tmpG, (size_t)64 * DBAT_GSZ);
    AL(h->d_partial, plan_partials(pl, up));
    AL(h->d_scal, SC_N);
    AL(h->d_x, P.n); AL(h->d_t, P.n); AL(h->d_p, P.n); AL(h->d_pgn, P.n); AL(h->d_g, P.n);
    AL(h->d_diagN, P.n); AL(h->d_dscale, P.n);
    AL(h->d_pEO, (size_t)6 * std::max(1, nImg) + 2);
    AL(h->d_r, pl.m);
    if (cudaMallocHost((void**)&h->h_scal, sizeof(double) * SC_N) != cudaSuccess ||
        cudaMallocHost((void**)&h->h_G, sizeof(double) * DBAT_GSZ) != cudaSuccess ||
        cudaMallocHost((void**)&h->h_piv, sizeof(unsigned long long) * 4) != cudaSuccess)
        return fail_create(h, DBAT_E_OOM, "cudaMallocHost failed");
    h->ev.resize(4096);
    for (auto& e : h->ev) cudaEventCreate(&e);
    cudaMemset(h->d_p, 0, sizeof(double) * P.n);
    if (cudaDeviceSynchronize() != cudaSuccess) return fail_create(h, DBAT_E_CUDA, "device error during create");
    if (!g_in_group_create) h->dcopy = copy_desc(d, pl.NC);
    *out = h;
    return DBAT_OK;
}

extern "C" void dbat_destroy(dbat_handle* h) {
    if (!h) return;
    if (h->group) group_destroy(h);
    if (h->dcopy) { free_desc(h->dcopy); h->dcopy = nullptr; }
    if (h->st) cudaStreamSynchronize(h->st);
    for (void* p : h->allocs) cudaFree(p);
    if (h->h_scal) cudaFreeHost(h->h_scal);
    if (h->h_G) cudaFreeHost(h->h_G);
    if (h->h_piv) cudaFreeHost(h->h_piv);
    tchol_free(h->tc);
    for (auto& e : h->ev) cudaEventDestroy(e);
    if (h->comm && g_nccl.CommDestroy) g_nccl.CommDestroy(h->comm);
    if (h->st2) cudaStreamDestroy(h->st2);
    if (h->evFork) cudaEventDestroy(h->evFork);
    if (h->evJoin) cudaEventDestroy(h->evJoin);
    if (h->evStep) cudaEventDestroy(h->evStep);
    if (h->st) cudaStreamDestroy(h->st);
    delete h;
}
extern "C" const char* dbat_last_error(const dbat_handle* h) { return h ? h->err.c_str() : g_create_err.c_str(); }
extern "C" int64_t dbat_num_unknowns(const dbat_handle* h) { return h ? h->P.n : 0; }
extern "C" int64_t dbat_num_residuals(const dbat_handle* h) { return h ? h->plan.m : 0; }
extern "C" int dbat_reduced_info(const dbat_handle* h, int64_t* info) {
    if (!h || !info) return DBAT_E_BADARG;
    if (h->group) h = group_first(h);
    const TileSym& s = h->tc.sym;
    const int64_t v[16] = {s.nT, s.ld, s.nS, s.nSlots, s.nSlotsS, s.nTasks, s.nTerms, s.depth, s.order_mode, s.nSeg,
                           h->tc.gridFactor, h->tc.gridBwd, h->P.nPsbig, h->P.nBig, h->P.grpMaxRays, h->plan.grpMaxPts};
    memcpy(info, v, sizeof(v));
    return DBAT_OK;
}

// --------------------------------------------------------------------------------------------
// evaluation building blocks
// --------------------------------------------------------------------------------------------
static int allreduce(dbat_handle* h, double* buf, size_t cnt) {
    if (h->nranks <= 1) return 0;
    int rc = g_nccl.AllReduce(buf, buf, cnt, /*ncclDouble*/ 8, /*ncclSum*/ 0, h->comm, h->st);
    if (rc != 0) { h->err = std::string("ncclAllReduce: ") + (g_nccl.GetErrorString ? g_nccl.GetErrorString(rc) : "?"); return DBAT_E_NCCL; }
    return 0;
}

static int nccl_fail(dbat_handle* h, const char* what, int rc) {
    h->err = std::string(what) + ": " + (g_nccl.GetErrorString ? g_nccl.GetErrorString(rc) : "?");
    return DBAT_E_NCCL;
}
// every part's own tiles of S end up, summed over the ranks, on the rank that factors them
static int reduce_owned_tiles(dbat_handle* h) {
    TChol& tc = h->tc;
    int rc = g_nccl.GroupStart();
    if (rc) return nccl_fail(h, "ncclGroupStart", rc);
    for (int g = 0; g < tc.sym.nParts && !rc; ++g) {
        const size_t b = tc.sym.ownSBegin[g], e = tc.sym.ownSBegin[g + 1];
        if (e > b) rc = g_nccl.Reduce(tc.d.tiles + b * TC_TT, tc.d.tiles + b * TC_TT, (e - b) * TC_TT, /*ncclDouble*/ 8, /*ncclSum*/ 0, g, h->comm, h->st);
    }
    const int rc2 = g_nccl.GroupEnd();
    if (rc) return nccl_fail(h, "ncclReduce", rc);
    if (rc2) return nccl_fail(h, "ncclGroupEnd", rc2);
    return 0;
}
static int allreduce_max_u64(dbat_handle* h, unsigned long long* buf, size_t cnt) {
    int rc = g_nccl.AllReduce(buf, buf, cnt, /*ncclUint64*/ 5, /*ncclMax*/ 2, h->comm, h->st);
    return rc ? nccl_fail(h, "ncclAllReduce", rc) : 0;
}

// scatter device vector xdev into the parameter arrays and rebuild the per-image records
static void set_params(dbat_handle* h, const double* xdev) {
    launch_set_params(h->P, xdev, ScatterList{h->d_IOsrc, h->d_IOdst, h->P.IOval, h->nIOdes, 0},
                      ScatterList{h->d_EOsrc, h->d_EOdst, h->P.EOval, h->nEOdes, 0},
                      ScatterList{h->d_OPsrc, h->d_OPdst, h->P.OPval, h->nOPdes, 0}, h->d_rep, h->plan.nIOrec, h->st);
}

static inline double gram_host(const double* G, int R, int C) {
    if (R < C) std::swap(R, C);
    const int p = R >> 3, q = C >> 3, i = R & 7, j = C & 7;
    return G[(p * (p + 1) / 2 + q) * 64 + (i * 4 + (j >> 1)) * 2 + (j & 1)];
}

// host-side end of eval_full once the stream has been synchronised: h_scal[SC_RR] = r'r (global)
static int finish_eval(dbat_handle* h) {
    h->h_scal[SC_RR] = gram_host(h->h_G, DBAT_COL_R, DBAT_COL_R) + h->h_scal[SC_PRR];
    h->normal_valid = true;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { h->err = std::string("eval_full: ") + cudaGetErrorString(e); return DBAT_E_CUDA; }
    return 0;
}

// residual + Jacobian + assembly at d_x.  On return h_scal[SC_RR] = r'r (global).  sync = false: everything is only
// queued on the stream (no host round trip); the caller synchronises later and calls finish_eval.
static int eval_full(dbat_handle* h, bool sync = true) {
    size_t a = ph_begin(h);
    h->cscWeighted = -1;                    // any cached Jacobian export belongs to an older x
    h->jp_vec = nullptr;
    set_params(h, h->d_x);
    h->params_valid = true;
    // camera side and point side read the same parameters and write disjoint outputs; both are latency- rather than
    // bandwidth-bound, so they run side by side on two streams
    // The camera-side kernel (the shorter one) is launched first: the two kernels cannot share an SM's registers, so they
    // run one after the other anyway, and this way the chunk -> image -> total sums run beside the point side.  Capping
    // the camera-side CTAs per SM to make room for point-side CTAs was measured and is slower.
    cudaEventRecord(h->evFork, h->st);
    cudaStreamWaitEvent(h->st2, h->evFork, 0);
    launch_cam_side(h->P, h->d_img_chunk_start, h->d_tmpG, h->st);
    launch_point_side(h->P, h->st2);
    cudaEventRecord(h->evJoin, h->st2);
    cudaStreamWaitEvent(h->st, h->evJoin, 0);
    const bool clearPrior = h->nranks > 1;      // the in-place allreduce below leaves the sums of all ranks in these arrays
    launch_prior_apply(h->P, h->d_x, h->d_camDiag, h->d_camG, h->d_col2pt, clearPrior, h->st);
    // r'r = Gram(r,r) + prior rows
    double* hG = h->h_G;
    launch_prior_rr(h->P, h->d_x, h->d_partial, h->d_prr, 0, clearPrior, h->st);
    if (h->nranks > 1) {
        // camera-side sums are partial per rank (each rank holds a subset of the points): one allreduce
        int rc = allreduce(h, h->d_evalRed, h->nEvalRed);
        if (rc) return rc;
    }
    cudaMemcpyAsync(hG, h->P.shG, sizeof(double) * DBAT_GSZ, cudaMemcpyDeviceToHost, h->st);
    cudaMemcpyAsync(h->h_scal + SC_PRR, h->d_prr, sizeof(double), cudaMemcpyDeviceToHost, h->st);
    ph_end(h, PH_EVAL, a);
    if (!sync) return 0;
    cudaStreamSynchronize(h->st);
    return finish_eval(h);
}

// weighted r'r at device vector xdev (residual only)
static int eval_rr(dbat_handle* h, const double* xdev, double* rr, bool sync = true) {
    size_t a = ph_begin(h);
    set_params(h, xdev);
    h->params_valid = (xdev == h->d_x);
    launch_resid(h->P, xdev, h->d_partial, h->d_scal, SC_RR, nullptr, 1, h->st);
    if (h->nranks > 1) { int rc = allreduce(h, h->d_scal + SC_RR, 1); if (rc) return rc; }
    cudaMemcpyAsync(h->h_scal + SC_RRT, h->d_scal + SC_RR, sizeof(double), cudaMemcpyDeviceToHost, h->st);   // own slot: SC_RR keeps r'r at d_x
    ph_end(h, PH_TRIAL, a);
    if (!sync) return 0;                        // the caller reads h_scal[SC_RRT] after its own synchronisation
    cudaError_t e = cudaStreamSynchronize(h->st);
    if (e != cudaSuccess) { h->err = std::string("eval_rr: ") + cudaGetErrorString(e); return DBAT_E_CUDA; }
    *rr = h->h_scal[SC_RRT];
    return 0;
}

// |J v|^2 and r'(J v) with J, r at d_x
static int eval_jp(dbat_handle* h, const double* v, double* jp2, double* rjp) {
    if (v == h->jp_vec && v) { *jp2 = h->jp_cache[0]; *rjp = h->jp_cache[1]; return 0; }   // by-product of solve_step
    size_t a = ph_begin(h);
    if (!h->params_valid) { set_params(h, h->d_x); h->params_valid = true; }
    launch_jp(h->P, h->d_x, v, h->d_partial, h->d_scal, SC_JP2, SC_RJP, h->st);
    if (h->nranks > 1) { int rc = allreduce(h, h->d_scal + SC_JP2, 2); if (rc) return rc; }
    cudaMemcpyAsync(h->h_scal + SC_JP2, h->d_scal + SC_JP2, 2 * sizeof(double), cudaMemcpyDeviceToHost, h->st);
    ph_end(h, PH_JP, a);
    cudaError_t e = cudaStreamSynchronize(h->st);
    if (e != cudaSuccess) { h->err = std::string("eval_jp: ") + cudaGetErrorString(e); return DBAT_E_CUDA; }
    *jp2 = h->h_scal[SC_JP2]; *rjp = h->h_scal[SC_RJP];
    return 0;
}

// dot product of two vectors in x layout.  With several ranks the camera part [0,nC) is
// replicated and the point part [nC,n) is distributed (zero outside the owned columns).
static int dev_dot(dbat_handle* h, const double* a, const double* b, int n, double* out) {
    if (h->nranks > 1 && n == h->P.n) {
        const int nC = h->P.nC;
        launch_dot(a, b, nC, h->d_partial, h->d_scal, SC_A, h->st);
        launch_dot(a + nC, b ? b + nC : nullptr, n - nC, h->d_partial, h->d_scal, SC_B, h->st);
        int rc = allreduce(h, h->d_scal + SC_B, 1);
        if (rc) return rc;
        cudaMemcpyAsync(h->h_scal + SC_A, h->d_scal + SC_A, 2 * sizeof(double), cudaMemcpyDeviceToHost, h->st);
        if (cudaStreamSynchronize(h->st) != cudaSuccess) { h->err = "dot failed"; return DBAT_E_CUDA; }
        *out = h->h_scal[SC_A] + h->h_scal[SC_B];
        return 0;
    }
    launch_dot(a, b, n, h->d_partial, h->d_scal, SC_A, h->st);
    cudaMemcpyAsync(h->h_scal + SC_A, h->d_scal + SC_A, sizeof(double), cudaMemcpyDeviceToHost, h->st);
    if (cudaStreamSynchronize(h->st) != cudaSuccess) { h->err = "dot failed"; return DBAT_E_CUDA; }
    *out = h->h_scal[SC_A];
    return 0;
}

// With several ranks a rank owns the camera part of x and its own points; the entries of other ranks' points in an
// uploaded vector are zeroed so that norms and dot products add up over the ranks.
__global__ void k_mask_unowned(double* __restrict__ x, const int* __restrict__ col2pt, int nC, int n) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (nC + k < n && col2pt[k] < 0) x[nC + k] = 0.0;
}
static void mask_unowned(dbat_handle* h, double* x) {
    if (h->nranks <= 1 || h->P.n <= h->P.nC) return;
    k_mask_unowned<<<(h->P.n - h->P.nC + 255) / 256, 256, 0, h->st>>>(x, h->d_col2pt, h->P.nC, h->P.n);
    count_launch();
}

// host-side end of solve_step once the stream has been synchronised
static void finish_solve(dbat_handle* h, int* singular) {
    // MATLAB's mldivide warns (singularMatrix / nearlySingularMatrix) when rcond < eps; with the
    // Cholesky factor rcond ~ (min pivot / max pivot)^2.
    double mm[2];
    memcpy(mm, h->h_piv, sizeof(mm));
    const int info = (int)h->h_piv[2];
    h->jp_cache[0] = h->h_scal[SC_JPP] + h->h_scal[SC_JPP + 2];
    h->jp_cache[1] = h->h_scal[SC_JPP + 1] + h->h_scal[SC_JPP + 3];
    h->jp_vec = h->solve_pout;
    const double ratio = mm[1] > 0 ? mm[0] / mm[1] : 1.0;      // no camera-side unknown at all: nothing to be singular
    *singular = (info != 0) || !(ratio * ratio > 2.220446049250313e-16);
}

// Solve the (damped, optionally Jacobi-scaled) normal equations at d_x -> step in `pout`.
// singular: 1 if the reduced system was not positive definite / numerically singular.
// sync = false: queued only; the caller synchronises the stream later and calls finish_solve.
static int solve_step(dbat_handle* h, double lambda, bool jacobi, double* pout, int* singular, bool sync = true) {
    DevProblem& P = h->P;
    TChol& tc = h->tc;
    size_t a = ph_begin(h);
    launch_build_S(P, h->d_camDiag, h->d_camG, lambda, h->st);
    if (h->nranks > 1 && h->rank != 0) {
        // only rank 0 contributes N_cc + lambda*I and -g_c; the others add their Schur terms to zero
        tchol_zero(tc, h->st);
        cudaMemsetAsync(P.rhs, 0, sizeof(double) * P.ldS, h->st);
    }
    launch_schur(P, lambda, h->st);
    const bool dist = h->nranks > 1 && tc.sym.nParts > 1;
    if (h->nranks > 1) {
        int rc;
        if (dist) rc = reduce_owned_tiles(h);        // top tiles are summed later, together with the partial factor updates
        else rc = allreduce(h, tc.d.tiles, (size_t)tc.d.nTopS * TC_TT);      // one contiguous array: no packing
        if (!rc) rc = allreduce(h, P.rhs, P.ldS);
        if (rc) return rc;
    }
    if (jacobi) {
        launch_diag(P, h->d_camDiag, h->d_diagN, h->st);
        launch_inv_sqrt(h->d_diagN, h->d_dscale, P.nC, h->st);
        launch_scale_prep(P, h->d_dscale, h->d_dS, h->st);
        tchol_scale(tc, h->d_dS, h->st);
    }
    ph_end(h, PH_SCHUR, a);
    a = ph_begin(h);
    tchol_put_rhs(tc, P.rhs, h->st, !dist || h->rank == 0);
    static const char* profPath = getenv("DBAT_TCHOL_PROF");       // debugging: per-task time stamps of the 3rd factorisation
    static int profCount = 0;
    unsigned long long* dprof = nullptr;
    if (profPath && ++profCount == 3) { cudaMalloc(&dprof, sizeof(unsigned long long) * 4 * tc.sym.nTasks); cudaMemset(dprof, 0, sizeof(unsigned long long) * 4 * tc.sym.nTasks); tc.d.prof = dprof; }
    tchol_factor_begin(tc, h->st);
    if (dist) {
        // every rank has factored the columns of its own subtree and subtracted its subtree's contribution from the
        // separator ("top") tiles: sum them, then everybody factors the top
        int rc = allreduce(h, tc.d.tiles, (size_t)tc.d.nTop * TC_TT);
        if (rc) return rc;
    }
    tchol_factor_end(tc, h->st);
    if (dprof) {
        cudaStreamSynchronize(h->st);
        const TileSym& sy = tc.sym;
        std::vector<unsigned long long> hp((size_t)4 * sy.nTasks);
        cudaMemcpy(hp.data(), dprof, sizeof(unsigned long long) * hp.size(), cudaMemcpyDeviceToHost);
        unsigned long long t0 = ~0ull;
        for (int t = 0; t < sy.nTasks; ++t) if (hp[4 * t]) t0 = std::min(t0, hp[4 * t]);
        if (FILE* f = fopen(profPath, "w")) {
            fprintf(f, "task,I,J,level,mode,nterms,t_claim,t_terms,t_deps,t_end\n");
            for (int t = 0; t < sy.nTasks; ++t)
                fprintf(f, "%d,%d,%d,%d,%d,%lld,%lld,%lld,%lld,%lld\n", t, sy.taskI[t], sy.taskJ[t], sy.level[sy.taskJ[t]], (int)sy.taskMode[t],
                        (long long)(sy.termPtr[t + 1] - sy.termPtr[t]), (long long)(hp[4 * t] - t0), (long long)(hp[4 * t + 1] - t0),
                        (long long)(hp[4 * t + 2] - t0), (long long)(hp[4 * t + 3] - t0));
            fclose(f);
        }
        cudaFree(dprof); tc.d.prof = nullptr;
    }
    ph_end(h, PH_CHOL, a);
    a = ph_begin(h);
    tchol_solve(tc, h->st);
    if (dist) {
        tchol_solve_owned_mask(tc, h->rank == 0, h->st);
        int rc = allreduce(h, tc.xs, P.ldS);
        if (!rc) { tchol_pack_stats(tc, h->d_stats, false, h->st); rc = allreduce_max_u64(h, h->d_stats, 3); tchol_pack_stats(tc, h->d_stats, true, h->st); }
        if (rc) return rc;
    }
    launch_unpermute(P, tc.xs, jacobi ? h->d_dscale : nullptr, h->d_pc, h->d_pEO, h->st);
    double* jpOut = h->d_scal + SC_JPP;
    launch_backsub(P, lambda, h->d_pc, h->d_pEO, pout, h->d_partial, h->d_camDiag, h->d_camG, jpOut, h->st, h->st2, h->evFork, h->evJoin);
    if (h->nranks > 1) { int rc = allreduce(h, jpOut, 2); if (rc) return rc; }     // point parts; the camera part is global already
    cudaMemcpyAsync(h->h_scal + SC_JPP, jpOut, 4 * sizeof(double), cudaMemcpyDeviceToHost, h->st);
    // pivot statistics into pinned memory (a copy into pageable memory would block the host until it has run)
    h->h_piv[2] = 0;
    cudaMemcpyAsync(h->h_piv + 2, tc.d.info, sizeof(int), cudaMemcpyDeviceToHost, h->st);
    cudaMemcpyAsync(h->h_piv, tc.d.minmax, 2 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, h->st);
    ph_end(h, PH_SOLVE, a);
    h->solve_pout = pout;
    h->jp_vec = nullptr;
    if (!sync) return 0;
    cudaError_t e = cudaStreamSynchronize(h->st);
    if (e != cudaSuccess) { h->err = std::string("solve_step: ") + cudaGetErrorString(e); return DBAT_E_CUDA; }
    finish_solve(h, singular);
    return 0;
}

// full gradient g = J'r into d_g (camera part from the Grams, point part from the records)
__global__ void k_gradient(DevProblem P, const double* __restrict__ camG, double* __restrict__ g);

// --------------------------------------------------------------------------------------------
// public evaluation entry points
// --------------------------------------------------------------------------------------------
extern "C" int dbat_eval(dbat_handle* h, const double* x, double* r, int weighted) {
    if (!h || !x) return DBAT_E_BADARG;
    if (h->group) return group_eval(h, x, r, weighted);
    CK(cudaMemcpyAsync(h->d_x, x, sizeof(double) * h->P.n, cudaMemcpyHostToDevice, h->st));
    set_params(h, h->d_x);
    h->params_valid = true; h->normal_valid = false; h->cscWeighted = -1;
    launch_resid(h->P, h->d_x, h->d_partial, h->d_scal, SC_RR, h->d_r, weighted, h->st);
    if (r) CK(cudaMemcpyAsync(r, h->d_r, sizeof(double) * h->plan.m, cudaMemcpyDeviceToHost, h->st));
    CK(cudaStreamSynchronize(h->st));
    return DBAT_OK;
}

static int build_csc(dbat_handle* h, int weighted) {
    if (h->cscWeighted == weighted) return 0;
    // several ranks: every rank exports the rows of ITS observations (and its prior rows); columns are x columns
    DevProblem& P = h->P;
    if (!h->params_valid) { set_params(h, h->d_x); h->params_valid = true; }
    const int LD = DBAT_NSLOT + 9;
    double* dJ = nullptr;
    const size_t cnt = (size_t)std::max(1, P.nObs) * 2 * LD;
    CK(cudaMalloc(&dJ, sizeof(double) * cnt));
    launch_export_jac(P, dJ, weighted, h->st);
    std::vector<double> J(cnt);
    cudaError_t e = cudaMemcpyAsync(J.data(), dJ, sizeof(double) * cnt, cudaMemcpyDeviceToHost, h->st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(h->st);
    cudaFree(dJ);
    if (e != cudaSuccess) { h->err = std::string("export: ") + cudaGetErrorString(e); return DBAT_E_CUDA; }
    // column -> (kind, index)
    const int n = P.n, nC = P.nC;
    std::vector<int> kind(n, -1), idx(n, -1);
    std::vector<std::vector<int>> ioUsers(n);   // IO column -> (image * NSLOT + slot) of every image that uses it, ascending
    for (int i = 0; i < P.nImg; ++i)
        for (int s = 0; s < DBAT_NSLOT; ++s) {
            const int c = h->plan.io_colx[(size_t)i * DBAT_NSLOT + s];
            if (c >= 0) { kind[c] = 0; ioUsers[c].push_back(i * DBAT_NSLOT + s); }
        }
    for (int e2 = 0; e2 < 6 * P.nImg; ++e2) if (h->plan.eo_col[e2] >= 0) { kind[h->plan.eo_col[e2]] = 1; idx[h->plan.eo_col[e2]] = e2; }
    for (int e2 = 0; e2 < 3 * P.nOP; ++e2) if (h->plan.op_col[e2] >= 0) { kind[h->plan.op_col[e2]] = 2; idx[h->plan.op_col[e2]] = e2; }
    std::vector<std::vector<int>> priorOfCol;   // rows of prior observations per column (rare)
    std::map<int, std::vector<int>> priorMap;
    for (int k = 0; k < P.nPrior; ++k) priorMap[h->plan.prior_col[k]].push_back(k);
    h->cscJc.assign(n + 1, 0); h->cscIr.clear(); h->cscV.clear();
    h->cscIr.reserve((size_t)P.nObs * 2 * 18); h->cscV.reserve((size_t)P.nObs * 2 * 18);
    auto push = [&](int64_t row, double v) { if (v != 0.0) { h->cscIr.push_back(row); h->cscV.push_back(v); } };
    (void)nC;
    for (int c = 0; c < n; ++c) {
        if (kind[c] == 0) {
            for (int u : ioUsers[c]) {                        // the observations of every image that uses the column
                const int i = u / DBAT_NSLOT, s = u % DBAT_NSLOT;
                for (int k = h->plan.img_start[i]; k < h->plan.img_start[i + 1]; ++k) {
                    push(2 * (int64_t)k, J[((size_t)k * 2) * LD + s]);
                    push(2 * (int64_t)k + 1, J[((size_t)k * 2 + 1) * LD + s]);
                }
            }
        } else if (kind[c] == 1) {
            const int i = idx[c] / 6, a2 = idx[c] % 6;
            for (int k = h->plan.img_start[i]; k < h->plan.img_start[i + 1]; ++k) {
                push(2 * (int64_t)k, J[((size_t)k * 2) * LD + DBAT_NSLOT + a2]);
                push(2 * (int64_t)k + 1, J[((size_t)k * 2 + 1) * LD + DBAT_NSLOT + a2]);
            }
        } else if (kind[c] == 2) {
            const int j = idx[c] / 3, t = idx[c] % 3;
            for (int o = h->plan.pt_start[j]; o < h->plan.pt_start[j + 1]; ++o) {
                const int k = h->plan.pm2cm[o];
                push(2 * (int64_t)k, J[((size_t)k * 2) * LD + DBAT_NSLOT + 6 + t]);
                push(2 * (int64_t)k + 1, J[((size_t)k * 2 + 1) * LD + DBAT_NSLOT + 6 + t]);
            }
        }
        auto it = priorMap.find(c);
        if (it != priorMap.end())
            for (int k : it->second) push(2 * (int64_t)P.nObs + k, weighted ? h->plan.prior_isig[k] : 1.0);
        h->cscJc[c + 1] = (int64_t)h->cscIr.size();
    }
    h->cscWeighted = weighted;
    return 0;
}
extern "C" int dbat_jacobian_nnz(dbat_handle* h, int weighted, int64_t* nnz) {
    if (!h || !nnz) return DBAT_E_BADARG;
    if (h->group) { h->err = "Jacobian export of a multi-device handle is not built: export from a single-device handle"; return DBAT_E_UNSUPPORTED; }
    int rc = build_csc(h, weighted ? 1 : 0);
    if (rc) return rc;
    *nnz = (int64_t)h->cscIr.size();
    return DBAT_OK;
}
extern "C" int dbat_jacobian_csc(dbat_handle* h, int weighted, int64_t* Jc, int64_t* Ir, double* vals) {
    if (!h || !Jc || !Ir || !vals) return DBAT_E_BADARG;
    if (h->group) { h->err = "Jacobian export of a multi-device handle is not built: export from a single-device handle"; return DBAT_E_UNSUPPORTED; }
    int rc = build_csc(h, weighted ? 1 : 0);
    if (rc) return rc;
    memcpy(Jc, h->cscJc.data(), sizeof(int64_t) * h->cscJc.size());
    memcpy(Ir, h->cscIr.data(), sizeof(int64_t) * h->cscIr.size());
    memcpy(vals, h->cscV.data(), sizeof(double) * h->cscV.size());
    return DBAT_OK;
}

extern "C" int dbat_normal_step(dbat_handle* h, const double* x, double lambda, int flags, double* p,
                                double* stats) {
    // flags: bit0 Jacobi scaling, bit1 also evaluate the trial point x+p, bit2 accept it when f decreases
    if (!h) return DBAT_E_BADARG;
    if (h->group) return group_normal_step(h, x, lambda, flags, p, stats);
    ph_reset(h);
    const size_t tot = ph_begin(h);
    if (x) { CK(cudaMemcpyAsync(h->d_x, x, sizeof(double) * h->P.n, cudaMemcpyHostToDevice, h->st)); h->cscWeighted = -1; mask_unowned(h, h->d_x); }
    const int64_t l0 = g_dbat_launches;
    // The whole iteration is queued without a host round trip; one synchronisation at the end, then the host-side
    // parts of the three stages.
    int rc = eval_full(h, false);
    if (rc) return rc;
    int sing = 0;
    rc = solve_step(h, lambda, (flags & 1) != 0, h->d_p, &sing, false);
    if (rc) return rc;
    double jp2 = 0, rjp = 0, fNew = NAN, rrT = 0;
    // the step goes back to the host on the second stream, beside the trial-point residual (queued after it in host
    // order: a pageable destination makes the copy call block)
    const bool sideCopy = p && (flags & 2);
    if (sideCopy) cudaEventRecord(h->evStep, h->st);
    else if (p) CK(cudaMemcpyAsync(p, h->d_p, sizeof(double) * h->P.n, cudaMemcpyDeviceToHost, h->st));
    if (flags & 2) {
        launch_axpy(1.0, h->d_p, h->d_x, h->d_t, h->P.n, h->st);
        rc = eval_rr(h, h->d_t, &rrT, false);
        if (rc) return rc;
    }
    if (sideCopy) {
        cudaStreamWaitEvent(h->st2, h->evStep, 0);
        CK(cudaMemcpyAsync(p, h->d_p, sizeof(double) * h->P.n, cudaMemcpyDeviceToHost, h->st2));
    }
    cudaError_t e = cudaStreamSynchronize(h->st);
    if (e == cudaSuccess && sideCopy) e = cudaStreamSynchronize(h->st2);
    if (e != cudaSuccess) { h->err = std::string("dbat_normal_step: ") + cudaGetErrorString(e); return DBAT_E_CUDA; }
    if ((rc = finish_eval(h))) return rc;
    finish_solve(h, &sing);
    rrT = h->h_scal[SC_RRT];
    const double f = 0.5 * h->h_scal[SC_RR];
    const bool jpCached = h->jp_vec == h->d_p;      // otherwise eval_jp sets the parameter arrays back to d_x
    rc = eval_jp(h, h->d_p, &jp2, &rjp);
    if (rc) return rc;
    if (flags & 2) {
        fNew = 0.5 * rrT;
        if ((flags & 4) && fNew < f) { std::swap(h->d_x, h->d_t); h->params_valid = jpCached; h->normal_valid = false; h->cscWeighted = -1; }
    }
    ph_end(h, PH_TOTAL, tot);
    ph_collect(h);
    if (stats) {
        stats[0] = f; stats[1] = jp2; stats[2] = rjp; stats[3] = sing; stats[4] = (double)(g_dbat_launches - l0);
        stats[5] = fNew; stats[6] = h->phase_ms[PH_TOTAL];
    }
    return DBAT_OK;
}

extern "C" int dbat_phase_times(const dbat_handle* h, const char** names, double* ms, int64_t* count, int cap) {
    if (!h) return 0;
    if (h->group) h = group_first(h);
    int n = std::min(cap, (int)PH_N);
    for (int i = 0; i < n; ++i) { if (names) names[i] = kPhaseNames[i]; if (ms) ms[i] = h->phase_ms[i]; if (count) count[i] = h->phase_cnt[i]; }
    return n;
}

// --------------------------------------------------------------------------------------------
// optimisers
// --------------------------------------------------------------------------------------------
extern "C" void dbat_default_opts(int method, dbat_opts* o) {
    if (!o) return;
    memset(o, 0, sizeof(*o));
    o->maxIter = 20; o->convTol = 1e-6; o->absTerm = 0; o->singularTest = 1; o->doTrace = 0;
    o->lambda0 = -1e-10; o->lambdaMin = -1e-10;           // bundle.m:301-304
    o->delta0 = -1.0;                                     // norm(x0), bundle.m:325
    o->alphaMin = 1e-9;                                   // bundle.m:283
    if (method == DBAT_METHOD_LMP) { o->mu = 0.25; o->eta = 0.75; }   // bundle.m:321-322
    else { o->mu = 0.1; o->eta = 0.0; }                   // bundle.m:281
}

struct TraceOut {
    dbat_result* res; int n; int cap;
    void store_x(dbat_handle* h, int col) {
        if (res->trace && col < cap)
            cudaMemcpyAsync(res->trace + (size_t)col * n, h->d_x, sizeof(double) * n, cudaMemcpyDeviceToHost, h->st);
        if (col + 1 > res->nTrace) res->nTrace = std::min(col + 1, cap);
    }
};

static bool term_fun(const dbat_opts* o, double jp2, double rr) {
    // bundle.m:186-192
    if (o->absTerm) return std::sqrt(rr) <= o->convTol;
    return std::sqrt(jp2) <= o->convTol * std::sqrt(rr);
}

// sprank(J) < n (levenberg_marquardt.m:126-135, gauss_newton_armijo.m:132-143): maximum bipartite
// matching between the columns and rows of the sparse Jacobian (exact zeros dropped, like the
// reference's J).  The device exports only the non-zero PATTERN of the per-observation blocks (8 bytes per
// observation); the adjacency of a column is enumerated from the problem's own index structure - all
// observations for a shared IO column, the image's for an EO column, the point's for an OP column, plus prior
// rows - so no CSC matrix is ever formed and the exact test runs at any size.  Greedy initialisation +
// augmenting paths (iterative DFS).
static bool matching_deficient(dbat_handle* h) {
    DevProblem& P = h->P;
    if (!h->params_valid) { set_params(h, h->d_x); h->params_valid = true; }
    const int n = P.n, m = h->plan.m, nObs = P.nObs;
    const int LD = DBAT_NSLOT + 9;
    std::vector<unsigned long long> mask(std::max(1, nObs));
    {
        unsigned long long* dm = nullptr;
        if (cudaMalloc(&dm, sizeof(unsigned long long) * mask.size()) != cudaSuccess) return false;
        launch_export_mask(P, dm, h->st);
        cudaError_t e = cudaMemcpyAsync(mask.data(), dm, sizeof(unsigned long long) * mask.size(), cudaMemcpyDeviceToHost, h->st);
        if (e == cudaSuccess) e = cudaStreamSynchronize(h->st);
        cudaFree(dm);
        if (e != cudaSuccess) return false;
    }
    // column -> (kind, index)
    std::vector<int> kind(n, -1), idx(n, -1);
    std::vector<std::vector<int>> ioUsers(n);            // IO column -> image * NSLOT + slot, images ascending
    std::vector<std::vector<int64_t>> ioCum(n);          // ... and the running count of their observations
    for (int i = 0; i < P.nImg; ++i)
        for (int s = 0; s < DBAT_NSLOT; ++s) {
            const int c = h->plan.io_colx[(size_t)i * DBAT_NSLOT + s];
            if (c < 0) continue;
            kind[c] = 0;
            ioUsers[c].push_back(i * DBAT_NSLOT + s);
            ioCum[c].push_back((ioCum[c].empty() ? 0 : ioCum[c].back()) + (h->plan.img_start[i + 1] - h->plan.img_start[i]));
        }
    for (int e2 = 0; e2 < 6 * P.nImg; ++e2) if (h->plan.eo_col[e2] >= 0) { kind[h->plan.eo_col[e2]] = 1; idx[h->plan.eo_col[e2]] = e2; }
    for (int e2 = 0; e2 < 3 * P.nOP; ++e2) if (h->plan.op_col[e2] >= 0) { kind[h->plan.op_col[e2]] = 2; idx[h->plan.op_col[e2]] = e2; }
    std::vector<std::vector<int>> priorRows(n);
    for (int k = 0; k < P.nPrior; ++k) priorRows[h->plan.prior_col[k]].push_back(2 * nObs + k);
    // adjacency of column c: position pos in [0, deg(c)) -> row or -1 (entry is an exact zero)
    auto degree = [&](int c) -> int64_t {
        int64_t d = (int64_t)priorRows[c].size();
        if (kind[c] == 0) d += 2 * (ioCum[c].empty() ? 0 : ioCum[c].back());
        else if (kind[c] == 1) { const int i = idx[c] / 6; d += 2 * (int64_t)(h->plan.img_start[i + 1] - h->plan.img_start[i]); }
        else if (kind[c] == 2) { const int j = idx[c] / 3; d += 2 * (int64_t)(h->plan.pt_start[j + 1] - h->plan.pt_start[j]); }
        return d;
    };
    auto row_at = [&](int c, int64_t pos) -> int {
        int64_t nb = degree(c) - (int64_t)priorRows[c].size();
        if (pos >= nb) return priorRows[c][(size_t)(pos - nb)];
        const int r = (int)(pos & 1);
        int k, slot;
        if (kind[c] == 0) {
            const int64_t q = pos >> 1;
            const size_t u = (size_t)(std::upper_bound(ioCum[c].begin(), ioCum[c].end(), q) - ioCum[c].begin());
            const int i = ioUsers[c][u] / DBAT_NSLOT;
            k = h->plan.img_start[i] + (int)(q - (u ? ioCum[c][u - 1] : 0)); slot = ioUsers[c][u] % DBAT_NSLOT;
        }
        else if (kind[c] == 1) { k = h->plan.img_start[idx[c] / 6] + (int)(pos >> 1); slot = DBAT_NSLOT + idx[c] % 6; }
        else { k = h->plan.pm2cm[h->plan.pt_start[idx[c] / 3] + (int)(pos >> 1)]; slot = DBAT_NSLOT + 6 + idx[c] % 3; }
        return ((mask[k] >> (LD * r + slot)) & 1ull) ? 2 * k + r : -1;
    };
    std::vector<int> matchRow(m, -1), matchCol(n, -1), stamp(m, -1);
    int matched = 0;
    for (int c = 0; c < n; ++c) {                                // greedy pass
        const int64_t d = degree(c);
        for (int64_t pos = 0; pos < d; ++pos) {
            const int r = row_at(c, pos);
            if (r >= 0 && matchRow[r] < 0) { matchRow[r] = c; matchCol[c] = r; ++matched; break; }
        }
    }
    std::vector<int> stackCol; std::vector<int64_t> stackPos, stackDeg; std::vector<int> pathRow;
    for (int c0 = 0; c0 < n && matched < n; ++c0) {
        if (matchCol[c0] >= 0) continue;
        // iterative DFS for an augmenting path starting at the free column c0
        stackCol.assign(1, c0); stackPos.assign(1, 0); stackDeg.assign(1, degree(c0)); pathRow.clear();
        bool found = false;
        while (!stackCol.empty() && !found) {
            const int c = stackCol.back();
            int64_t& pos = stackPos.back();
            if (pos >= stackDeg.back()) { stackCol.pop_back(); stackPos.pop_back(); stackDeg.pop_back(); if (!pathRow.empty()) pathRow.pop_back(); continue; }
            const int r = row_at(c, pos++);
            if (r < 0 || stamp[r] == c0) continue;
            stamp[r] = c0;
            if (matchRow[r] < 0) { pathRow.push_back(r); found = true; break; }
            pathRow.push_back(r);
            const int c2 = matchRow[r];
            stackCol.push_back(c2); stackPos.push_back(0); stackDeg.push_back(degree(c2));
        }
        if (found) {                                              // flip the path: column k takes row pathRow[k]
            for (size_t k = 0; k < stackCol.size(); ++k) { matchRow[pathRow[k]] = stackCol[k]; matchCol[stackCol[k]] = pathRow[k]; }
            ++matched;
        }
    }
    return matched < n;
}

// counting screen (necessary conditions of a full structural rank): every unknown needs at least
// one residual row, every point/image needs as many rows as free coordinates, and m >= n.
static bool structurally_deficient(dbat_handle* h) {
    DevProblem& P = h->P;
    if (h->nranks > 1) return false;
    if (h->plan.m < P.n) return true;
    std::vector<int> priorCnt(P.n, 0);
    for (int c : h->plan.prior_col) priorCnt[c]++;
    for (int j = 0; j < P.nOP; ++j) {
        int freec = 0, pri = 0;
        for (int t = 0; t < 3; ++t) { const int c = h->plan.op_col[3 * (size_t)j + t]; if (c >= 0) { ++freec; pri += priorCnt[c]; } }
        if (freec && 2 * (h->plan.pt_start[j + 1] - h->plan.pt_start[j]) + pri < freec) return true;
    }
    for (int i = 0; i < P.nImg; ++i) {
        int freec = 0, pri = 0;
        for (int a = 0; a < 6; ++a) { const int c = h->plan.eo_col[6 * (size_t)i + a]; if (c >= 0) { ++freec; pri += priorCnt[c]; } }
        if (freec && 2 * (h->plan.img_start[i + 1] - h->plan.img_start[i]) + pri < freec) return true;
    }
    static const bool skipExact = getenv("DBAT_NO_SPRANK") != nullptr;
    if (skipExact) return false;
    return matching_deficient(h);          // exact at any size: 8 bytes per observation cross the bus
}

static int trace_sum(dbat_handle* h, double* tr) {
    cudaMemsetAsync(h->d_diagN, 0, sizeof(double) * h->P.n, h->st);
    launch_diag(h->P, h->d_camDiag, h->d_diagN, h->st);
    return dev_dot(h, h->d_diagN, nullptr, h->P.n, tr);
}

static int solve_lm(dbat_handle* h, const dbat_opts* o, dbat_result* res, TraceOut& T) {
    // levenberg_marquardt.m:54-247
    DevProblem& P = h->P;
    const int nn = P.n;
    int n = 0, code = 0, rc;
    if ((rc = eval_full(h))) return rc;                               // :76-82
    double rr = h->h_scal[SC_RR], f = 0.5 * rr;
    double lambda0 = o->lambda0, lambdaMin = o->lambdaMin;
    if (lambda0 < 0 || lambdaMin < 0) {                               // :88-95
        double tr = 0; if ((rc = trace_sum(h, &tr))) return rc;
        if (lambda0 < 0) lambda0 = std::fabs(lambda0) * tr / nn;
        if (lambdaMin < 0) lambdaMin = std::fabs(lambdaMin) * tr / nn;
    }
    double lambda = lambda0;
    if (lambda < lambdaMin) lambda = 0.0;
    res->nDamping = 0; res->nRr = 0;
    res->damping[res->nDamping++] = lambda;                           // :106
    double prevLambda = NAN, jp2 = 0, rjp = 0;
    const int cap = o->maxIter + 2;
    while (true) {
        while (n <= o->maxIter) {                                     // :117
            int sing = 0;
            // after the first iteration the solve and the trial-point residual are queued back to back and the host
            // waits once (LM never looks at the singular flag; the |Jp| statistics come out of the back-substitution)
            const bool defer = n > 0;
            if ((rc = solve_step(h, lambda, false, h->d_p, &sing, !defer))) return rc;   // :119
            if (res->nRr < cap + 1) res->rr[res->nRr++] = std::sqrt(rr);      // :122
            if (n == 0 && structurally_deficient(h)) {                // :126-135 (p = NaN)
                code = -4; cudaMemsetAsync(h->d_p, 0xff, sizeof(double) * nn, h->st); break;
            }
            if (res->nDamping < cap + 1) res->damping[res->nDamping++] = lambda;   // :136
            if (o->doTrace) printf("Levenberg-Marquardt: iteration %d, residual norm=%.2g, lambda=%.2g\n", n, std::sqrt(rr), lambda);
            T.store_x(h, n);                                          // :149-156
            n++;                                                      // :159
            if (!defer && (rc = eval_jp(h, h->d_p, &jp2, &rjp))) return rc;     // :162
            launch_axpy(1.0, h->d_p, h->d_x, h->d_t, nn, h->st);      // :165 t=x+p
            double rrNew = 0;
            if ((rc = eval_rr(h, h->d_t, &rrNew))) return rc;         // :166-167
            if (defer) {
                finish_solve(h, &sing);
                if ((rc = eval_jp(h, h->d_p, &jp2, &rjp))) return rc; // :162
            }
            const double fNew = 0.5 * rrNew;
            if (fNew < f) {                                           // :177 (no veto function)
                std::swap(h->d_x, h->d_t);
                lambda = lambda / 10;                                 // :181
                if (lambda < lambdaMin) lambda = 0.0;
                if ((rc = eval_full(h))) return rc;                   // :188-194
                rr = h->h_scal[SC_RR]; f = 0.5 * rr;
                break;
            } else {
                lambda = (lambda == 0.0) ? lambdaMin : lambda * 10;   // :198-206
            }
        }
        if (code != 0) break;
        if (prevLambda == 0.0 && term_fun(o, jp2, rr)) break;         // :217
        prevLambda = lambda;                                          // :222
        if (n > o->maxIter) { code = -1; break; }
    }
    T.store_x(h, n);                                                  // :238-240
    if (res->nRr < cap + 1) res->rr[res->nRr++] = std::sqrt(rr);      // :242
    res->code = code; res->iters = n;
    return 0;
}

static int solve_gna(dbat_handle* h, const dbat_opts* o, dbat_result* res, TraceOut& T) {
    // gauss_newton_armijo.m:75-290
    DevProblem& P = h->P;
    const int nn = P.n;
    int n = 0, code = 0, rc;
    const int cap = o->maxIter + 2;
    res->nDamping = 0; res->nRr = 0;
    T.store_x(h, 0);                                                  // :82
    double rr = 0;
    while (true) {
        if ((rc = eval_full(h))) return rc;                           // :112-116
        rr = h->h_scal[SC_RR];
        if (res->nRr < cap + 1) res->rr[res->nRr++] = std::sqrt(rr);
        if (o->doTrace) printf("Gauss-Newton-Armijo: iteration %d, residual norm=%.2g\n", n, std::sqrt(rr));
        if (n == 0 && structurally_deficient(h)) {                    // :132-143
            code = -4; cudaMemsetAsync(h->d_p, 0xff, sizeof(double) * nn, h->st); break;
        }
        int sing = 0;
        if ((rc = solve_step(h, 0.0, true, h->d_p, &sing))) return rc;   // :166-174
        if (o->singularTest && sing) { code = -2; break; }            // :176-184
        double jp2 = 0, rjp = 0;
        if ((rc = eval_jp(h, h->d_p, &jp2, &rjp))) return rc;         // :187
        if (term_fun(o, jp2, rr)) break;                              // :191
        n++;
        // linesearch (:249-290)
        const double f0 = 0.5 * rr, fp0 = rjp;
        double alpha = 1.0; bool found = false; double rrT = rr;
        while (alpha >= o->alphaMin) {
            launch_axpy(alpha, h->d_p, h->d_x, h->d_t, nn, h->st);
            if ((rc = eval_rr(h, h->d_t, &rrT))) return rc;
            if (0.5 * rrT < f0 + o->mu * alpha * fp0) { found = true; break; }
            alpha /= 2;
        }
        if (found) { std::swap(h->d_x, h->d_t); rr = rrT; h->params_valid = true; h->normal_valid = false; }
        else { alpha = 0.0; h->params_valid = false; }
        if (res->nDamping < cap + 1) res->damping[res->nDamping++] = alpha;
        T.store_x(h, n);
        if (alpha == 0.0) { code = -3; if (res->nRr < cap + 1) { res->rr[res->nRr] = res->rr[res->nRr - 1]; res->nRr++; } break; }   // :217-223
        if (n > o->maxIter) { code = -1; if (res->nRr < cap + 1) res->rr[res->nRr++] = std::sqrt(rr); break; }   // :225-231
    }
    res->code = code; res->iters = n;
    res->nTrace = std::min(n + 1, cap);
    return 0;
}

static int solve_gm(dbat_handle* h, const dbat_opts* o, dbat_result* res, TraceOut& T) {
    // gauss_markov.m:35-110: undamped Gauss-Newton, p = (J'J)\(-J'r), x = x + p; terminates on
    // norm(J p) <= convTol norm(r) (always the relative test, :86); no structural-rank test.
    DevProblem& P = h->P;
    const int nn = P.n;
    int n = 0, code = 0, rc;
    const int cap = o->maxIter + 2;
    res->nDamping = 0; res->nRr = 0;
    T.store_x(h, 0);                                                  // :42
    while (true) {
        if ((rc = eval_full(h))) return rc;                           // :58-61
        const double rr = h->h_scal[SC_RR];
        if (res->nRr < cap + 1) res->rr[res->nRr++] = std::sqrt(rr);  // :63
        if (o->doTrace) printf("Gauss-Markov: iteration %d, residual norm=%.2g\n", n, std::sqrt(rr));
        int sing = 0;
        // :69.  Solved with Jacobi column scaling (the same step p = D (D N D)^-1 D (-g)): the pivot-ratio
        // test that stands in for MATLAB's singular-matrix warning is only meaningful on the scaled system
        if ((rc = solve_step(h, 0.0, true, h->d_p, &sing))) return rc;
        if (o->singularTest && sing) { code = -2; break; }            // :71-79
        double jp2 = 0, rjp = 0;
        if ((rc = eval_jp(h, h->d_p, &jp2, &rjp))) return rc;
        if (std::sqrt(jp2) <= o->convTol * std::sqrt(rr)) break;      // :86
        n++;                                                          // :92
        launch_axpy(1.0, h->d_p, h->d_x, h->d_t, nn, h->st);          // :95
        std::swap(h->d_x, h->d_t);
        h->params_valid = false; h->normal_valid = false;
        T.store_x(h, n);                                              // :97-104
        if (n > o->maxIter) { code = -1; break; }                     // :107-110
    }
    res->code = code; res->iters = n;
    res->nTrace = std::min(n + 1, cap);
    return 0;
}

__global__ void k_gradient(DevProblem P, const double* __restrict__ camG, double* __restrict__ g) {
    // g = J'r : shared IO from the summed Gram, EO from the per-image Grams, OP from the records
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    auto gat = [](const double* G, int R, int C) {
        if (R < C) { const int q = R; R = C; C = q; }
        const int p = R >> 3, q = C >> 3, i = R & 7, j = C & 7;
        return G[(p * (p + 1) / 2 + q) * 64 + (i * 4 + (j >> 1)) * 2 + (j & 1)];
    };
    if (t < DBAT_NSLOT) { const int c = P.sh_col[t]; if (c >= 0) g[c] = gat(P.shG, t, DBAT_COL_R) + camG[c]; }
    if (t < 6 * P.nImg) {
        const int c = P.eo_col[t];
        if (c >= 0) g[c] = gat(P.imgG + (size_t)(t / 6) * DBAT_GSZ, DBAT_COL_EO + t % 6, DBAT_COL_R) + camG[c];
    }
    if (t < 3 * P.nOP) { const int c = P.op_col[t]; if (c >= 0) g[c] = P.pt[(size_t)(t / 3) * DBAT_PT_STRIDE + 6 + t % 3]; }
}

static int solve_lmp(dbat_handle* h, const dbat_opts* o, dbat_result* res, TraceOut& T) {
    // levenberg_marquardt_powell.m:60-335
    DevProblem& P = h->P;
    const int nn = P.n;
    int n = 0, code = 0, rc;
    const int cap = o->maxIter + 2;
    res->nDamping = 0; res->nRr = 0; res->nRhos = 0;
    double delta = o->delta0;
    if (!(delta > 0)) { double xx = 0; if ((rc = dev_dot(h, h->d_x, h->d_x, nn, &xx))) return rc; delta = std::sqrt(xx); }   // bundle.m:325
    if ((rc = eval_full(h))) return rc;                               // :95-99
    double rr = h->h_scal[SC_RR], f = 0.5 * rr;
    int ntr = 0;
    while (true) {
        if (res->nRr < cap + 1) res->rr[res->nRr++] = std::sqrt(rr);  // :109
        if (n == 0 && structurally_deficient(h)) {                    // :113-122 (p = NaN)
            code = -4; cudaMemsetAsync(h->d_p, 0xff, sizeof(double) * nn, h->st); break;
        }
        // dogleg (:232-335)
        int sing = 0, step = 0;
        if ((rc = solve_step(h, 0.0, true, h->d_pgn, &sing))) return rc;
        double pgn2 = 0; if ((rc = dev_dot(h, h->d_pgn, h->d_pgn, nn, &pgn2))) return rc;
        const double npGN = std::sqrt(pgn2);
        double jp2 = 0, rjp = 0;
        if (npGN <= delta) {                                          // :281-286
            cudaMemcpyAsync(h->d_p, h->d_pgn, sizeof(double) * nn, cudaMemcpyDeviceToDevice, h->st);
            step = 0;
        } else {
            int nt = std::max(std::max(3 * P.nOP, 6 * P.nImg), DBAT_NSLOT);
            cudaMemsetAsync(h->d_g, 0, sizeof(double) * nn, h->st);
            if (P.ioGeneral) {          // IO columns: prior part, then the sums over the images that use the column
                cudaMemcpyAsync(h->d_g, h->d_camG, sizeof(double) * P.nC, cudaMemcpyDeviceToDevice, h->st);
                launch_io_diag_grad_gen(P, nullptr, nullptr, nullptr, h->d_g, h->st);
            }
            k_gradient<<<(nt + 255) / 256, 256, 0, h->st>>>(P, h->d_camG, h->d_g); count_launch();
            double gg = 0, jg2 = 0, dummy = 0;
            if ((rc = dev_dot(h, h->d_g, h->d_g, nn, &gg))) return rc;
            if ((rc = eval_jp(h, h->d_g, &jg2, &dummy))) return rc;
            const double lambdaStar = gg / jg2;                       // :309  (g'Hg = |J g|^2)
            const double nCP = lambdaStar * std::sqrt(gg);
            if (nCP > delta) {                                        // :313-318
                cudaMemsetAsync(h->d_p, 0, sizeof(double) * nn, h->st);
                launch_axpy(-delta / std::sqrt(gg), h->d_g, h->d_p, h->d_p, nn, h->st);
                step = 2;
            } else {                                                  // :324-332
                double gp = 0; if ((rc = dev_dot(h, h->d_g, h->d_pgn, nn, &gp))) return rc;
                // CP = -ls*g ;  A=|CP-pGN|^2, B=2 CP.(pGN-CP), C=|CP|^2-delta^2
                const double cp2 = lambdaStar * lambdaStar * gg, cpp = -lambdaStar * gp;
                const double A = cp2 - 2 * cpp + pgn2, B = 2 * (cpp - cp2), C = cp2 - delta * delta;
                const double k = (-B + std::sqrt(B * B - 4 * A * C)) / (2 * A);
                // p = CP + k (pGN - CP) = (1-k)(-ls) g + k pGN
                cudaMemsetAsync(h->d_p, 0, sizeof(double) * nn, h->st);
                launch_axpy(k, h->d_pgn, h->d_p, h->d_p, nn, h->st);
                launch_axpy(-(1 - k) * lambdaStar, h->d_g, h->d_p, h->d_p, nn, h->st);
                step = 1;
            }
        }
        if (res->nDamping < cap + 1) res->damping[res->nDamping++] = delta;   // :128
        if (res->steps && n < cap) res->steps[n] = step;
        if ((rc = eval_jp(h, h->d_p, &jp2, &rjp))) return rc;         // :131-132
        if (step == 0 && term_fun(o, jp2, rr)) break;                 // :134
        launch_axpy(1.0, h->d_p, h->d_x, h->d_t, nn, h->st);          // :143
        double rrT = 0;
        if ((rc = eval_rr(h, h->d_t, &rrT))) return rc;
        const double ft = 0.5 * rrT;
        const double predicted = -rjp - 0.5 * jp2;                    // :153
        const double actual = f - ft;
        const double rho = actual / predicted;
        if (res->rhos && res->nRhos < cap) res->rhos[res->nRhos] = rho;
        res->nRhos++;
        if (o->doTrace) printf("Levenberg-Marquardt-Powell: iteration %d, residual norm=%.2g, delta=%.2g, step=%d, rho=%.1f\n", n, std::sqrt(rr), delta, step, rho);
        if (rho <= o->mu) {                                           // :166-179 (a NaN rho is not <= mu: accepted, like the reference)
            delta = delta / 2;
            if (delta > npGN) delta = delta / std::exp2(std::ceil(std::log2(delta / npGN)));
        } else {                                                      // :180-195
            std::swap(h->d_x, h->d_t);
            if ((rc = eval_full(h))) return rc;
            rr = h->h_scal[SC_RR]; f = 0.5 * rr;
            if (rho >= o->eta) delta = delta * 2;
        }
        T.store_x(h, n);                                              // :197-204 T(:,n+1)=x
        ntr = n + 1;
        n++;
        if (n > o->maxIter) { code = -1; break; }
    }
    res->code = code; res->iters = n;
    res->nTrace = std::min(ntr, n);                                   // :226 T=T(:,1:n)
    if (res->nRhos > cap) res->nRhos = cap;
    return 0;
}

extern "C" int dbat_solve(dbat_handle* h, int method, const dbat_opts* opts, const double* x0, dbat_result* res) {
    if (!h || !opts || !x0 || !res || !res->x || !res->rr || !res->damping) return DBAT_E_BADARG;
    if (h->group) return group_solve(h, method, opts, x0, res);
    const int nn = h->P.n;
    CK(cudaMemcpyAsync(h->d_x, x0, sizeof(double) * nn, cudaMemcpyHostToDevice, h->st));
    mask_unowned(h, h->d_x);
    CK(cudaMemsetAsync(h->d_p, 0, sizeof(double) * nn, h->st));
    CK(cudaMemsetAsync(h->d_pgn, 0, sizeof(double) * nn, h->st));
    CK(cudaMemsetAsync(h->d_g, 0, sizeof(double) * nn, h->st));
    CK(cudaMemsetAsync(h->d_t, 0, sizeof(double) * nn, h->st));
    h->cscWeighted = -1; h->params_valid = false; h->normal_valid = false;
    ph_reset(h);
    const int64_t l0 = g_dbat_launches;
    res->nTrace = 0; res->code = 0; res->iters = 0; res->nRhos = 0;
    TraceOut T{res, nn, opts->maxIter + 2};
    auto t0 = std::chrono::steady_clock::now();
    int rc;
    switch (method) {
        case DBAT_METHOD_GM: rc = solve_gm(h, opts, res, T); break;
        case DBAT_METHOD_LM: rc = solve_lm(h, opts, res, T); break;
        case DBAT_METHOD_GNA: rc = solve_gna(h, opts, res, T); break;
        case DBAT_METHOD_LMP: rc = solve_lmp(h, opts, res, T); break;
        default: h->err = "unknown method"; return DBAT_E_BADARG;
    }
    if (rc) return rc;
    CK(cudaStreamSynchronize(h->st));
    res->seconds = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    res->launches = g_dbat_launches - l0;
    // final outputs
    CK(cudaMemcpyAsync(res->x, h->d_x, sizeof(double) * nn, cudaMemcpyDeviceToHost, h->st));
    if (res->p) CK(cudaMemcpyAsync(res->p, h->d_p, sizeof(double) * nn, cudaMemcpyDeviceToHost, h->st));
    if (res->r_w || res->r_u) {
        set_params(h, h->d_x); h->params_valid = true;
        if (res->r_w) {
            launch_resid(h->P, h->d_x, h->d_partial, h->d_scal, SC_PRR, h->d_r, 1, h->st);
            CK(cudaMemcpyAsync(res->r_w, h->d_r, sizeof(double) * h->plan.m, cudaMemcpyDeviceToHost, h->st));
            CK(cudaStreamSynchronize(h->st));
        }
        if (res->r_u) {
            launch_resid(h->P, h->d_x, h->d_partial, h->d_scal, SC_PRR, h->d_r, 0, h->st);
            CK(cudaMemcpyAsync(res->r_u, h->d_r, sizeof(double) * h->plan.m, cudaMemcpyDeviceToHost, h->st));
        }
    }
    ph_collect(h);
    CK(cudaStreamSynchronize(h->st));
    return DBAT_OK;
}

// --------------------------------------------------------------------------------------------
// posterior covariance (bundle_cov.m): everything from the undamped reduced system
//   C_cam = inv(S) ;  COP_j = V_j^-1 + V_j^-1 W~_j' C_cam W~_j V_j^-1   (SURVEY.md §3.4)
// --------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) k_cop(DevProblem P, const double* __restrict__ C, int ldc,
                                              const double* __restrict__ dsc, double s02, double* __restrict__ out);


// ---- full point covariances (bundle_cov 'CXX' / 'COPF').  With T_j[a] = (V_j^-1 w_a) for the camera-side
// rows a of point j (shared IO slots, then 6 per observation; w_a the 3-vector of the cross block):
//   U  = Ccc (B V^-1)            U[r, xc]  = sum_a Ccc[r, col(a)] T_j[a][t]        (nCam x nOPcols)
//   Cpp = V^-1 + (B V^-1)' U     Cpp[xc, xc'] = [j == j'] Vi[t][t'] + sum_a T_j[a][t] U[col(a), xc']
//   Ccp = -U
__global__ void k_cov_rows(DevProblem P, double* __restrict__ T, int* __restrict__ Tc) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= P.nOP) return;
    const size_t r0 = (size_t)DBAT_NSLOT * j + 6 * (size_t)P.pt_start[j];
    const int o0 = P.pt_start[j], k = P.pt_start[j + 1] - o0;
    const double* rec = P.pt + (size_t)j * DBAT_PT_STRIDE;
    const double* v = P.vinv + (size_t)j * 8;
    const double Vi[6] = {v[0], v[1], v[2], v[3], v[4], v[5]};
    for (int a = 0; a < DBAT_NSLOT + 6 * k; ++a) {
        const double* w; int col;
        if (a < DBAT_NSLOT) { w = rec + DBAT_PT_WSH + 3 * a; col = P.sh_s[a]; }
        else {
            const int o = (a - DBAT_NSLOT) / 6, e = (a - DBAT_NSLOT) % 6;
            w = P.W + (size_t)(o0 + o) * DBAT_W_STRIDE + 3 * e;
            col = P.eo_s[6 * (size_t)P.img_pm[o0 + o] + e];
        }
        double* t = T + 3 * (r0 + a);
        t[0] = Vi[0] * w[0] + Vi[1] * w[1] + Vi[2] * w[2];
        t[1] = Vi[1] * w[0] + Vi[3] * w[1] + Vi[4] * w[2];
        t[2] = Vi[2] * w[0] + Vi[4] * w[1] + Vi[5] * w[2];
        Tc[r0 + a] = col;
    }
}
// C and dsc are in S order (Tc holds S indices); U is indexed by x columns
__global__ void k_cov_U(DevProblem P, const double* __restrict__ C, int ldc, const double* __restrict__ dsc,
                        const double* __restrict__ T, const int* __restrict__ Tc, const int* __restrict__ x2s,
                        double* __restrict__ U) {
    const int rx = blockIdx.x * blockDim.x + threadIdx.x;
    if (rx >= P.nC) return;
    const int r = x2s[rx];
    const double dr = dsc[r];
    for (int j = blockIdx.y; j < P.nOP; j += gridDim.y) {       // gridDim.y stops at 65535, nOP does not
        const int* opc = P.op_col + 3 * (size_t)j;
        if (opc[0] < 0 && opc[1] < 0 && opc[2] < 0) continue;
        const size_t r0 = (size_t)DBAT_NSLOT * j + 6 * (size_t)P.pt_start[j];
        const int rows = DBAT_NSLOT + 6 * (P.pt_start[j + 1] - P.pt_start[j]);
        double u[3] = {0.0, 0.0, 0.0};
        for (int a = 0; a < rows; ++a) {
            const int ca = Tc[r0 + a];
            if (ca < 0) continue;
            const double c = C[(size_t)ca * ldc + r] * dr * dsc[ca];
            const double* t = T + 3 * (r0 + a);
            u[0] += c * t[0]; u[1] += c * t[1]; u[2] += c * t[2];
        }
        for (int t = 0; t < 3; ++t) if (opc[t] >= 0) U[(size_t)(opc[t] - P.nC) * P.nC + rx] = u[t];
    }
}
__global__ void k_cov_pp(DevProblem P, const double* __restrict__ T, const int* __restrict__ Tc,
                         const double* __restrict__ U, const int* __restrict__ col2pt, double* __restrict__ Cpp) {
    const int m3 = P.n - P.nC;
    const int xc = blockIdx.x * blockDim.x + threadIdx.x;      // column xc (point j'), row point j
    if (xc >= m3) return;
    const double* Uc = U + (size_t)xc * P.nC;
    const int code = col2pt[xc];                          // 3 j' + t' of OP column nC + xc
    for (int j = blockIdx.y; j < P.nOP; j += gridDim.y) {
        const int* opc = P.op_col + 3 * (size_t)j;
        if (opc[0] < 0 && opc[1] < 0 && opc[2] < 0) continue;
        const size_t r0 = (size_t)DBAT_NSLOT * j + 6 * (size_t)P.pt_start[j];
        const int rows = DBAT_NSLOT + 6 * (P.pt_start[j + 1] - P.pt_start[j]);
        double acc[3] = {0.0, 0.0, 0.0};
        for (int a = 0; a < rows; ++a) {
            const int ca = Tc[r0 + a];
            if (ca < 0) continue;
            const double u = Uc[P.s2x[ca]];
            const double* t = T + 3 * (r0 + a);
            acc[0] += t[0] * u; acc[1] += t[1] * u; acc[2] += t[2] * u;
        }
        if (code / 3 == j) {
            const double* v = P.vinv + (size_t)j * 8;
            const int tp = code % 3;
            const double Vrow[3][3] = {{v[0], v[1], v[2]}, {v[1], v[3], v[4]}, {v[2], v[4], v[5]}};
            acc[0] += Vrow[0][tp]; acc[1] += Vrow[1][tp]; acc[2] += Vrow[2][tp];
        }
        for (int t = 0; t < 3; ++t) if (opc[t] >= 0) Cpp[(size_t)xc * m3 + (opc[t] - P.nC)] = acc[t];
    }
}

__global__ void k_dense_unit_diag(double* __restrict__ A, int ld, int from) {
    const int k = from + blockIdx.x * blockDim.x + threadIdx.x;
    if (k < ld) A[(size_t)k * ld + k] = 1.0;
}
// undamped point blocks: numerically singular (relative pivot below 1e-13) -> *bad = 1
__global__ void k_point_pd_check(DevProblem P, int* __restrict__ bad) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= P.nOP) return;
    const int* opc = P.op_col + 3 * (size_t)j;
    const bool f0 = opc[0] >= 0, f1 = opc[1] >= 0, f2 = opc[2] >= 0;
    if (!f0 && !f1 && !f2) return;
    const double* rec = P.pt + (size_t)j * DBAT_PT_STRIDE;
    const double a00 = f0 ? rec[0] : 1.0, a11 = f1 ? rec[3] : 1.0, a22 = f2 ? rec[5] : 1.0;
    const double a01 = (f0 && f1) ? rec[1] : 0.0, a02 = (f0 && f2) ? rec[2] : 0.0, a12 = (f1 && f2) ? rec[4] : 0.0;
    const double tol = 1e-13;
    bool ok = a00 > 0.0;
    const double l10 = a01 / sqrt(a00), l20 = a02 / sqrt(a00);
    const double d1 = a11 - l10 * l10;
    ok = ok && d1 > tol * a11;
    const double l21 = (a12 - l20 * l10) / sqrt(d1);
    const double d2 = a22 - l20 * l20 - l21 * l21;
    ok = ok && d2 > tol * a22;
    if (!ok) *bad = 1;
}

// Common front of the covariance entry points: the undamped, Jacobi-scaled reduced system (tiles, S order) -> dense
// copy -> dense factor -> explicit inverse C (device, ld x ld, S order, of the SCALED system; h->d_dscale unscales).
// The dense path (chol.cu) is kept for the covariances: inv(S) is a full matrix.  *info != 0: not positive definite.
static int cov_factor(dbat_handle* h, double** Zp, double** Cp, int* ldp, int* infop) {
    // several ranks: every rank holds the whole (summed) reduced system and inverts it redundantly; CIO / CEO come out
    // identical everywhere, COP covers the points of this rank (it shards by point like the solve, bundle_cov.m:400-455)
    DevProblem& P = h->P;
    int rc;
    cudaGetLastError();                      // a launch error reported by this call is one of its own launches
    if (!h->normal_valid) { if ((rc = eval_full(h))) return rc; }
    launch_build_S(P, h->d_camDiag, h->d_camG, 0.0, h->st);
    if (h->nranks > 1 && h->rank != 0) { tchol_zero(h->tc, h->st); cudaMemsetAsync(P.rhs, 0, sizeof(double) * P.ldS, h->st); }
    launch_schur(P, 0.0, h->st);
    if (h->nranks > 1) {                     // every tile of S, summed, on every rank
        const TCholDev& td = h->tc.d;
        rc = allreduce(h, td.tiles, (size_t)td.nTopS * TC_TT);
        if (!rc && td.nOwnS > 0) rc = allreduce(h, td.tiles + (size_t)td.nTop * TC_TT, (size_t)td.nOwnS * TC_TT);
        if (rc) return rc;
    }
    launch_diag(P, h->d_camDiag, h->d_diagN, h->st);
    launch_inv_sqrt(h->d_diagN, h->d_dscale, P.nC, h->st);
    launch_scale_prep(P, h->d_dscale, h->d_dS, h->st);
    tchol_scale(h->tc, h->d_dS, h->st);
    const int ldd = (P.ldS + 127) / 128 * 128;
    double *Sd = nullptr, *Z = nullptr, *C = nullptr;
    const size_t sz = sizeof(double) * (size_t)ldd * ldd;
    int* d_bad = nullptr;
    CholWork cw;
    if (cudaMalloc(&Sd, sz) != cudaSuccess || cudaMalloc(&Z, sz) != cudaSuccess || cudaMalloc(&C, sz) != cudaSuccess ||
        cudaMalloc(&d_bad, sizeof(int)) != cudaSuccess || chol_alloc(cw, ldd)) {
        cudaFree(Sd); cudaFree(Z); cudaFree(C); cudaFree(d_bad);
        h->err = "out of memory for the covariance workspace"; return DBAT_E_OOM;
    }
    cudaMemsetAsync(Sd, 0, sz, h->st);
    cudaMemsetAsync(d_bad, 0, sizeof(int), h->st);
    tchol_to_dense(h->tc, Sd, ldd, h->st);
    k_dense_unit_diag<<<(ldd + 255) / 256, 256, 0, h->st>>>(Sd, ldd, P.ldS - 1);      // rhs row position and padding
    // a point block that is not positive definite (a point with a single ray) makes the reference's
    // factorisation of the full normal matrix fail (bundle_cov.m:87-107): report that, not huge numbers
    if (P.nOP > 0) k_point_pd_check<<<(P.nOP + 255) / 256, 256, 0, h->st>>>(P, d_bad);
    count_launch(2);
    chol_factor(cw, Sd, h->st);
    chol_inverse(cw, Sd, Z, C, h->st);
    // a failed launch leaves no trace a stream synchronisation reports: ask for it
    const cudaError_t le = cudaGetLastError();
    int info = 0, badPts = 0;
    cudaMemcpyAsync(&info, cw.info, sizeof(int), cudaMemcpyDeviceToHost, h->st);
    cudaMemcpyAsync(&badPts, d_bad, sizeof(int), cudaMemcpyDeviceToHost, h->st);
    cudaError_t e = cudaStreamSynchronize(h->st);
    if (e == cudaSuccess) e = le;
    chol_free(cw);
    cudaFree(Sd); cudaFree(d_bad);
    if (e != cudaSuccess) { cudaFree(Z); cudaFree(C); h->err = std::string("dbat_cov: ") + cudaGetErrorString(e); return DBAT_E_CUDA; }
    if (badPts) info = -1;
    *Zp = Z; *Cp = C; *ldp = ldd; *infop = info;
    return 0;
}

extern "C" int dbat_cov(dbat_handle* h, int which, double s0, double* out) {
    if (!h || !out) return DBAT_E_BADARG;
    if (h->group) return group_cov(h, which, s0, out);
    DevProblem& P = h->P;
    int rc;
    double *Z = nullptr, *C = nullptr;
    int ldd = 0, info = 0;
    if ((rc = cov_factor(h, &Z, &C, &ldd, &info))) return rc;
    const size_t sz = sizeof(double) * (size_t)ldd * ldd;
    cudaError_t e = cudaSuccess;
    const double s02 = s0 * s0;
    const int nC = P.nC, ld = ldd;
    const std::vector<int>& x2s = h->plan.x2s;
    if ((which == DBAT_COV_CXX || which == DBAT_COV_CXX_OP) && P.ioGeneral) {
        cudaFree(Z); cudaFree(C);
        h->err = "the dense point covariance (CXX / COPF) is built for one shared IO block only; use CIO / CEO / COP";
        return DBAT_E_UNSUPPORTED;
    }
    if (which == DBAT_COV_CXX || which == DBAT_COV_CXX_OP) {
        const int m3 = P.n - nC;
        const size_t limit = (size_t)1 << 28;                 // 2 GB of doubles per dense block
        if ((size_t)m3 * m3 > limit || (size_t)nC * m3 > limit || (which == DBAT_COV_CXX && (size_t)P.n * P.n > limit)) {
            cudaFree(Z); cudaFree(C);
            h->err = "dense point covariance too large (more than 2 GB); use COP for the 3x3 blocks";
            return DBAT_E_UNSUPPORTED;
        }
        const size_t nRows = (size_t)DBAT_NSLOT * P.nOP + 6 * (size_t)P.nObs;
        double *T = nullptr, *U = nullptr, *Cpp = nullptr; int *Tc = nullptr, *d_x2s = nullptr;
        if (cudaMalloc(&d_x2s, sizeof(int) * x2s.size()) ||
            cudaMemcpy(d_x2s, x2s.data(), sizeof(int) * x2s.size(), cudaMemcpyHostToDevice) ||
            cudaMalloc(&T, sizeof(double) * 3 * std::max<size_t>(1, nRows)) || cudaMalloc(&Tc, sizeof(int) * std::max<size_t>(1, nRows)) ||
            cudaMalloc(&U, sizeof(double) * std::max<size_t>(1, (size_t)nC * m3)) || cudaMalloc(&Cpp, sizeof(double) * std::max<size_t>(1, (size_t)m3 * m3))) {
            cudaFree(d_x2s); cudaFree(T); cudaFree(Tc); cudaFree(U); cudaFree(Cpp); cudaFree(Z); cudaFree(C);
            h->err = "out of memory for the point covariance"; return DBAT_E_OOM;
        }
        cudaMemsetAsync(U, 0, sizeof(double) * std::max<size_t>(1, (size_t)nC * m3), h->st);
        cudaMemsetAsync(Cpp, 0, sizeof(double) * std::max<size_t>(1, (size_t)m3 * m3), h->st);
        if (P.nOP > 0 && m3 > 0) {
            launch_point_vinv(P, 0.0, h->st);
            k_cov_rows<<<(P.nOP + 127) / 128, 128, 0, h->st>>>(P, T, Tc);
            const unsigned gy = (unsigned)std::min(P.nOP, 65535);
            k_cov_U<<<dim3((nC + 127) / 128, gy), 128, 0, h->st>>>(P, C, ld, h->d_dS, T, Tc, d_x2s, U);
            k_cov_pp<<<dim3((m3 + 127) / 128, gy), 128, 0, h->st>>>(P, T, Tc, U, h->d_col2pt, Cpp);
            count_launch(3);
        }
        const cudaError_t le = cudaGetLastError();
        std::vector<double> hpp((size_t)m3 * m3), hu, hc, dsc;
        cudaMemcpyAsync(hpp.data(), Cpp, sizeof(double) * hpp.size(), cudaMemcpyDeviceToHost, h->st);
        if (which == DBAT_COV_CXX) {
            hu.resize((size_t)nC * m3); hc.resize((size_t)ld * ld); dsc.resize(std::max(1, nC));
            cudaMemcpyAsync(hu.data(), U, sizeof(double) * hu.size(), cudaMemcpyDeviceToHost, h->st);
            cudaMemcpyAsync(hc.data(), C, sz, cudaMemcpyDeviceToHost, h->st);
            cudaMemcpyAsync(dsc.data(), h->d_dscale, sizeof(double) * nC, cudaMemcpyDeviceToHost, h->st);
        }
        e = cudaStreamSynchronize(h->st);
        if (e == cudaSuccess) e = le;
        cudaFree(d_x2s); cudaFree(T); cudaFree(Tc); cudaFree(U); cudaFree(Cpp);
        if (e != cudaSuccess) { cudaFree(Z); cudaFree(C); h->err = std::string("dbat_cov: ") + cudaGetErrorString(e); return DBAT_E_CUDA; }
        const double nanv = NAN;
        if (which == DBAT_COV_CXX_OP) {
            for (size_t k = 0; k < hpp.size(); ++k) out[k] = info != 0 ? nanv : s02 * hpp[k];
        } else {
            const size_t n = (size_t)P.n;
            for (size_t b = 0; b < n; ++b)
                for (size_t a = 0; a < n; ++a) {
                    double v;
                    if (a < (size_t)nC && b < (size_t)nC) v = hc[(size_t)x2s[b] * ld + x2s[a]] * dsc[a] * dsc[b];
                    else if (a < (size_t)nC) v = -hu[(b - nC) * nC + a];
                    else if (b < (size_t)nC) v = -hu[(a - nC) * nC + b];
                    else v = hpp[(b - nC) * m3 + (a - nC)];
                    out[b * n + a] = info != 0 ? nanv : s02 * v;
                }
        }
    } else if (which == DBAT_COV_COP) {
        double* dOut = nullptr;
        cudaMalloc(&dOut, sizeof(double) * 9 * (size_t)std::max(1, P.nOP));
        cudaMemsetAsync(dOut, 0, sizeof(double) * 9 * (size_t)std::max(1, P.nOP), h->st);
        if (P.nOP > 0 && P.ioGeneral) launch_cop_gen(P, C, ld, h->d_dS, s02, dOut, h->st);
        else if (P.nOP > 0) { k_cop<<<(P.nOP + 3) / 4, 128, 0, h->st>>>(P, C, ld, h->d_dS, s02, dOut); count_launch(); }
        const cudaError_t le = cudaGetLastError();
        cudaMemcpyAsync(out, dOut, sizeof(double) * 9 * (size_t)P.nOP, cudaMemcpyDeviceToHost, h->st);
        e = cudaStreamSynchronize(h->st);
        if (e == cudaSuccess) e = le;
        cudaFree(dOut);
    } else {
        // bring the camera covariance to the host and unscale: C = D Cs D
        std::vector<double> hc((size_t)ld * ld), dsc(std::max(1, nC));
        e = cudaMemcpy(hc.data(), C, sz, cudaMemcpyDeviceToHost);
        if (e == cudaSuccess) e = cudaMemcpy(dsc.data(), h->d_dscale, sizeof(double) * nC, cudaMemcpyDeviceToHost);
        if (e != cudaSuccess) { cudaFree(Z); cudaFree(C); h->err = std::string("dbat_cov: ") + cudaGetErrorString(e); return DBAT_E_CUDA; }
        auto cv = [&](int a, int b) { return (info != 0) ? NAN : s02 * hc[(size_t)x2s[b] * ld + x2s[a]] * dsc[a] * dsc[b]; };
        if (which == DBAT_COV_CXX_CAM) {
            for (int b = 0; b < nC; ++b) for (int a = 0; a < nC; ++a) out[(size_t)b * nC + a] = cv(a, b);
        } else if (which == DBAT_COV_CEO || which == DBAT_COV_CIO) {
            const int R = which == DBAT_COV_CEO ? 6 : h->plan.NC;
            const std::vector<int>& col = which == DBAT_COV_CEO ? h->plan.eo_col : h->plan.io_col;
            for (int i = 0; i < P.nImg; ++i)
                for (int b = 0; b < R; ++b)
                    for (int a = 0; a < R; ++a) {
                        const int ca = col[(size_t)i * R + a], cb = col[(size_t)i * R + b];
                        out[((size_t)i * R + b) * R + a] = (ca >= 0 && cb >= 0) ? cv(ca, cb) : 0.0;
                    }
        } else { cudaFree(Z); cudaFree(C); h->err = "unknown covariance selector"; return DBAT_E_BADARG; }
    }
    cudaFree(Z); cudaFree(C);
    if (e != cudaSuccess) { h->err = std::string("dbat_cov: ") + cudaGetErrorString(e); return DBAT_E_CUDA; }
    return info != 0 ? DBAT_E_NOTSPD : DBAT_OK;
}

// ---- report-side consumers of the covariance on the device (covstats.cu; SURVEY §8f N2)
int cov_block_stats(const double* d_blocks, const int* d_cols, int k, long long N, double thres, double* d_std_x,
                    long long cap, long long* nHits, long long* h_block, int* h_row, int* h_col, double* h_rho,
                    cudaStream_t st);
void launch_cam_blocks(const double* C, int ld, const int* x2s, const double* dsc, const int* cols, int k, long long N,
                       double s02, int bad, double* out, cudaStream_t st);
__global__ void k_cop(DevProblem P, const double* __restrict__ C, int ldc, const double* __restrict__ dsc, double s02,
                      double* __restrict__ out);

extern "C" int dbat_cov_stats(dbat_handle* h, double s0, double thres, double* std_x, dbat_cov_hit_list* io,
                              dbat_cov_hit_list* eo, dbat_cov_hit_list* op) {
    if (!h || !std_x) return DBAT_E_BADARG;
    if (h->group || h->nranks > 1) { h->err = "dbat_cov_stats runs on a single-device handle; use dbat_cov per rank"; return DBAT_E_UNSUPPORTED; }
    DevProblem& P = h->P;
    int rc;
    double *Z = nullptr, *C = nullptr;
    int ld = 0, info = 0;
    if ((rc = cov_factor(h, &Z, &C, &ld, &info))) return rc;
    cudaFree(Z);
    const double s02 = s0 * s0;
    const int NC = h->plan.NC, nImg = P.nImg;
    int *d_x2s = nullptr, *d_iocol = nullptr;
    double *d_std = nullptr, *d_blk = nullptr;
    const size_t nBlk = std::max<size_t>(std::max<size_t>((size_t)NC * NC * nImg, (size_t)36 * nImg), (size_t)9 * std::max(1, P.nOP));
    if (cudaMalloc(&d_x2s, sizeof(int) * std::max<size_t>(1, h->plan.x2s.size())) || cudaMalloc(&d_iocol, sizeof(int) * std::max<size_t>(1, h->plan.io_col.size())) ||
        cudaMalloc(&d_std, sizeof(double) * std::max(1, P.n)) || cudaMalloc(&d_blk, sizeof(double) * std::max<size_t>(1, nBlk))) {
        cudaFree(C); cudaFree(d_x2s); cudaFree(d_iocol); cudaFree(d_std); cudaFree(d_blk);
        h->err = "out of memory for the covariance statistics"; return DBAT_E_OOM;
    }
    cudaMemcpyAsync(d_x2s, h->plan.x2s.data(), sizeof(int) * h->plan.x2s.size(), cudaMemcpyHostToDevice, h->st);
    cudaMemcpyAsync(d_iocol, h->plan.io_col.data(), sizeof(int) * h->plan.io_col.size(), cudaMemcpyHostToDevice, h->st);
    cudaMemsetAsync(d_std, 0, sizeof(double) * std::max(1, P.n), h->st);
    int ce = 0;
    auto run = [&](const int* cols, int k, long long N, dbat_cov_hit_list* L) {
        long long nh = 0;
        dbat_cov_hit_list none = {0, 0, nullptr, nullptr, nullptr, nullptr};
        if (!L) L = &none;
        const int e1 = cov_block_stats(d_blk, cols, k, N, thres, d_std, (long long)L->cap, &nh, (long long*)L->block, L->row, L->col, L->rho, h->st);
        L->n = nh;
        if (e1 && !ce) ce = e1;
    };
    // IO: the NC x NC block of every image (images of one camera hold identical blocks), EO: 6 x 6 per image
    launch_cam_blocks(C, ld, d_x2s, h->d_dscale, d_iocol, NC, nImg, s02, info != 0, d_blk, h->st);
    run(d_iocol, NC, nImg, io);
    launch_cam_blocks(C, ld, d_x2s, h->d_dscale, P.eo_col, 6, nImg, s02, info != 0, d_blk, h->st);
    run(P.eo_col, 6, nImg, eo);
    // OP: 3 x 3 per point, as dbat_cov(COP) forms them
    cudaMemsetAsync(d_blk, 0, sizeof(double) * 9 * (size_t)std::max(1, P.nOP), h->st);
    if (P.nOP > 0 && P.ioGeneral) launch_cop_gen(P, C, ld, h->d_dS, s02, d_blk, h->st);
    else if (P.nOP > 0) { k_cop<<<(P.nOP + 3) / 4, 128, 0, h->st>>>(P, C, ld, h->d_dS, s02, d_blk); count_launch(); }
    run(P.op_col, 3, P.nOP, op);
    const cudaError_t le = cudaGetLastError();
    cudaMemcpyAsync(std_x, d_std, sizeof(double) * P.n, cudaMemcpyDeviceToHost, h->st);
    cudaError_t e = cudaStreamSynchronize(h->st);
    if (e == cudaSuccess) e = le;
    cudaFree(C); cudaFree(d_x2s); cudaFree(d_iocol); cudaFree(d_std); cudaFree(d_blk);
    if (e != cudaSuccess || ce) { h->err = std::string("dbat_cov_stats: ") + cudaGetErrorString(e != cudaSuccess ? e : (cudaError_t)ce); return DBAT_E_CUDA; }
    if (info != 0) { for (int c = 0; c < P.n; ++c) std_x[c] = NAN; return DBAT_E_NOTSPD; }
    return DBAT_OK;
}

// COP: one warp per point.  Row set of W~_j: shared IO slots (NSLOT) then 6 per observation.
// u_a = sum_b Cs[col_a,col_b] d_a d_b T_b ,  COP = Vi + sum_a T_a' u_a   with T_a = W_a Vi (1x3)
__global__ void __launch_bounds__(128) k_cop(DevProblem P, const double* __restrict__ C, int ldc,
                                              const double* __restrict__ dsc, double s02, double* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int j = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (j >= P.nOP) return;
    const int* opc = P.op_col + 3 * (size_t)j;
    if (opc[0] < 0 && opc[1] < 0 && opc[2] < 0) return;
    const double* rec = P.pt + (size_t)j * DBAT_PT_STRIDE;
    // Vi (undamped) — same arithmetic as point_inverse in schur.cu
    double a00 = rec[0], a01 = rec[1], a02 = rec[2], a11 = rec[3], a12 = rec[4], a22 = rec[5];
    const bool f0 = opc[0] >= 0, f1 = opc[1] >= 0, f2 = opc[2] >= 0;
    if (!f0) a00 = 1.0; if (!f1) a11 = 1.0; if (!f2) a22 = 1.0;
    const double l00 = sqrt(a00), l10 = a01 / l00, l20 = a02 / l00;
    const double l11 = sqrt(a11 - l10 * l10), l21 = (a12 - l20 * l10) / l11;
    const double l22 = sqrt(a22 - l20 * l20 - l21 * l21);
    const double m00 = 1.0 / l00, m11 = 1.0 / l11, m22 = 1.0 / l22;
    const double m10 = -l10 * m00 * m11, m21 = -l21 * m11 * m22, m20 = -(l20 * m00 + l21 * m10) * m22;
    double Vi[6] = {m00 * m00 + m10 * m10 + m20 * m20, m10 * m11 + m20 * m21, m20 * m22,
                    m11 * m11 + m21 * m21, m21 * m22, m22 * m22};
    if (!f0) { Vi[0] = 0; Vi[1] = 0; Vi[2] = 0; }
    if (!f1) { Vi[1] = 0; Vi[3] = 0; Vi[4] = 0; }
    if (!f2) { Vi[2] = 0; Vi[4] = 0; Vi[5] = 0; }
    const int o0 = P.pt_start[j], k = P.pt_start[j + 1] - o0;
    const int nRows = DBAT_NSLOT + 6 * k;
    auto row_col = [&](int a) -> int {                 // S index of row a
        if (a < DBAT_NSLOT) return P.sh_s[a];
        const int o = (a - DBAT_NSLOT) / 6, e = (a - DBAT_NSLOT) % 6;
        return P.eo_s[6 * (size_t)P.img_pm[o0 + o] + e];
    };
    auto row_T = [&](int a, double T[3]) {
        const double* w = (a < DBAT_NSLOT) ? rec + DBAT_PT_WSH + 3 * a
                                           : P.W + (size_t)(o0 + (a - DBAT_NSLOT) / 6) * DBAT_W_STRIDE + 3 * ((a - DBAT_NSLOT) % 6);
        T[0] = Vi[0] * w[0] + Vi[1] * w[1] + Vi[2] * w[2];
        T[1] = Vi[1] * w[0] + Vi[3] * w[1] + Vi[4] * w[2];
        T[2] = Vi[2] * w[0] + Vi[4] * w[1] + Vi[5] * w[2];
    };
    double acc[6] = {0, 0, 0, 0, 0, 0};
    for (int a = lane; a < nRows; a += 32) {
        const int ca = row_col(a);
        if (ca < 0) continue;
        double Ta[3]; row_T(a, Ta);
        double u[3] = {0, 0, 0};
        for (int b = 0; b < nRows; ++b) {
            const int cb = row_col(b);
            if (cb < 0) continue;
            double Tb[3]; row_T(b, Tb);
            const double c = C[(size_t)cb * ldc + ca] * dsc[ca] * dsc[cb];
            u[0] += c * Tb[0]; u[1] += c * Tb[1]; u[2] += c * Tb[2];
        }
        acc[0] += Ta[0] * u[0]; acc[1] += Ta[0] * u[1]; acc[2] += Ta[0] * u[2];
        acc[3] += Ta[1] * u[1]; acc[4] += Ta[1] * u[2]; acc[5] += Ta[2] * u[2];
    }
#pragma unroll
    for (int q = 0; q < 6; ++q)
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc[q] += __shfl_xor_sync(0xffffffffu, acc[q], o);
    if (lane == 0) {
        double* o9 = out + 9 * (size_t)j;
        const double c00 = s02 * (Vi[0] + acc[0]), c01 = s02 * (Vi[1] + acc[1]), c02 = s02 * (Vi[2] + acc[2]);
        const double c11 = s02 * (Vi[3] + acc[3]), c12 = s02 * (Vi[4] + acc[4]), c22 = s02 * (Vi[5] + acc[5]);
        o9[0] = c00; o9[1] = c01; o9[2] = c02; o9[3] = c01; o9[4] = c11; o9[5] = c12; o9[6] = c02; o9[7] = c12; o9[8] = c22;
    }
}

// --------------------------------------------------------------------------------------------
// stand-alone access to the dense factor + inverse of the covariances (unit tests, profiling)
// --------------------------------------------------------------------------------------------
extern "C" int dbat_dense_chol_inverse(int64_t n, const double* A, double* Ainv, int repeat, double* ms_out) {
    if (n <= 0 || !A || !Ainv) return DBAT_E_BADARG;
    // the layout cov_factor factors: room for the rhs row of S, identity padding
    const int ld = std::max(128, (int)((n + 1 + 127) / 128) * 128);
    const size_t sz = sizeof(double) * (size_t)ld * ld;
    std::vector<double> hA((size_t)ld * ld, 0.0);
    for (int64_t c = 0; c < n; ++c) for (int64_t r = 0; r < n; ++r) hA[(size_t)c * ld + r] = A[(size_t)c * n + r];
    for (int64_t k = n; k < ld; ++k) hA[(size_t)k * ld + k] = 1.0;
    double *dA0 = nullptr, *dA = nullptr, *Z = nullptr, *Cc = nullptr;
    CholWork w;
    cudaGetLastError();                      // a launch error reported by this call is one of its own launches
    if (cudaMalloc(&dA0, sz) || cudaMalloc(&dA, sz) || cudaMalloc(&Z, sz) || cudaMalloc(&Cc, sz) || chol_alloc(w, ld)) {
        cudaFree(dA0); cudaFree(dA); cudaFree(Z); cudaFree(Cc);
        g_create_err = "dbat_dense_chol_inverse: out of memory"; return DBAT_E_OOM;
    }
    cudaMemcpy(dA0, hA.data(), sz, cudaMemcpyHostToDevice);
    cudaStream_t st; cudaStreamCreate(&st);
    cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
    float best = 1e30f;
    for (int it = 0; it < std::max(1, repeat); ++it) {
        cudaMemcpyAsync(dA, dA0, sz, cudaMemcpyDeviceToDevice, st);
        cudaEventRecord(e0, st);
        chol_factor(w, dA, st);
        chol_inverse(w, dA, Z, Cc, st);
        cudaEventRecord(e1, st);
        cudaStreamSynchronize(st);
        float ms = 0; cudaEventElapsedTime(&ms, e0, e1); best = std::min(best, ms);
    }
    int info = 0;
    cudaMemcpy(&info, w.info, sizeof(int), cudaMemcpyDeviceToHost);
    cudaMemcpy(hA.data(), Cc, sz, cudaMemcpyDeviceToHost);
    for (int64_t c = 0; c < n; ++c) for (int64_t r = 0; r < n; ++r) Ainv[(size_t)c * n + r] = hA[(size_t)c * ld + r];
    if (ms_out) *ms_out = best;
    cudaError_t e = cudaDeviceSynchronize();
    if (e == cudaSuccess) e = cudaGetLastError();
    chol_free(w); cudaFree(dA0); cudaFree(dA); cudaFree(Z); cudaFree(Cc);
    cudaEventDestroy(e0); cudaEventDestroy(e1); cudaStreamDestroy(st);
    if (e != cudaSuccess) { g_create_err = std::string("dbat_dense_chol_inverse: ") + cudaGetErrorString(e); return DBAT_E_CUDA; }
    return info != 0 ? DBAT_E_NOTSPD : DBAT_OK;
}

// The sparse tile solver on a caller-supplied SPD matrix: blocks of 6 columns play the images.
extern "C" int dbat_tile_chol_solve(int64_t n, const double* A, const double* b, double* x, int64_t mode,
                                    int64_t leafImages, int repeat, double* stats) {
    if (n <= 0 || !A || !b || !x) return DBAT_E_BADARG;
    const int nImg = (int)((n + 5) / 6);
    std::vector<int> nEO(nImg, 6);
    nEO[nImg - 1] = (int)(n - 6 * (int64_t)(nImg - 1));
    std::vector<std::vector<int32_t>> nb(nImg);
    for (int64_t c = 0; c < n; ++c)
        for (int64_t r = c + 1; r < n; ++r)
            if (A[(size_t)c * n + r] != 0.0 && r / 6 != c / 6) { nb[r / 6].push_back((int32_t)(c / 6)); nb[c / 6].push_back((int32_t)(r / 6)); }
    std::vector<int64_t> ap(nImg + 1, 0); std::vector<int32_t> ad;
    for (int i = 0; i < nImg; ++i) {
        std::sort(nb[i].begin(), nb[i].end());
        nb[i].erase(std::unique(nb[i].begin(), nb[i].end()), nb[i].end());
        ap[i] = (int64_t)ad.size(); ad.insert(ad.end(), nb[i].begin(), nb[i].end());
    }
    ap[nImg] = (int64_t)ad.size();
    TileSym sym;
    if (tile_symbolic(nImg, ap.data(), ad.data(), nEO.data(), 0, (int)mode, (int)leafImages, sym)) return DBAT_E_BADARG;
    TChol tc;
    if (tchol_alloc(tc, sym)) { g_create_err = "dbat_tile_chol_solve: out of memory"; return DBAT_E_OOM; }
    // host tiles and rhs in S order
    std::vector<int> x2s(n);
    for (int64_t c = 0; c < n; ++c) x2s[c] = sym.imgS[c / 6] + (int)(c % 6);
    std::vector<double> ht((size_t)sym.nSlotsS * TC_TT, 0.0), hr(sym.ld, 0.0);
    for (int64_t c = 0; c < n; ++c)
        for (int64_t r = c; r < n; ++r) {
            const double v = A[(size_t)c * n + r];
            if (v == 0.0) continue;
            const int sr = std::max(x2s[r], x2s[c]), sc = std::min(x2s[r], x2s[c]);
            const int slot = sym.tix[(size_t)(sr / TC_T) * sym.nT + sc / TC_T];
            if (slot < 0 || slot >= sym.nSlotsS) { tchol_free(tc); g_create_err = "tile pattern misses an entry"; return DBAT_E_STATE; }
            ht[(size_t)slot * TC_TT + (sc % TC_T) * TC_T + sr % TC_T] = v;
        }
    for (int k = 0; k < sym.ld - 1; ++k)
        if (sym.s2kind[k] == 0) ht[(size_t)sym.tix[(size_t)(k / TC_T) * sym.nT + k / TC_T] * TC_TT + (k % TC_T) * TC_T + k % TC_T] = 1.0;
    for (int64_t c = 0; c < n; ++c) hr[x2s[c]] = b[c];
    double *d0 = nullptr, *drhs = nullptr;
    cudaMalloc(&d0, sizeof(double) * ht.size());
    cudaMalloc(&drhs, sizeof(double) * hr.size());
    cudaMemcpy(d0, ht.data(), sizeof(double) * ht.size(), cudaMemcpyHostToDevice);
    cudaMemcpy(drhs, hr.data(), sizeof(double) * hr.size(), cudaMemcpyHostToDevice);
    cudaStream_t st; cudaStreamCreate(&st);
    cudaEvent_t e0, e1, e2; cudaEventCreate(&e0); cudaEventCreate(&e1); cudaEventCreate(&e2);
    float best = 1e30f, bestF = 1e30f;
    const char* profPath = getenv("DBAT_TCHOL_PROF");        // per-task time stamps of the last repetition
    unsigned long long* dprof = nullptr;
    if (profPath) { cudaMalloc(&dprof, sizeof(unsigned long long) * 4 * sym.nTasks); tc.d.prof = dprof; }
    for (int it = 0; it < std::max(1, repeat); ++it) {
        cudaMemcpyAsync(tc.d.tiles, d0, sizeof(double) * ht.size(), cudaMemcpyDeviceToDevice, st);
        cudaEventRecord(e0, st);
        tchol_put_rhs(tc, drhs, st);
        tchol_factor(tc, st);
        cudaEventRecord(e2, st);
        tchol_solve(tc, st);
        cudaEventRecord(e1, st);
        cudaStreamSynchronize(st);
        float ms = 0; cudaEventElapsedTime(&ms, e0, e1); best = std::min(best, ms);
        cudaEventElapsedTime(&ms, e0, e2); bestF = std::min(bestF, ms);
    }
    if (profPath) {
        std::vector<unsigned long long> hp((size_t)4 * sym.nTasks);
        cudaMemcpy(hp.data(), dprof, sizeof(unsigned long long) * hp.size(), cudaMemcpyDeviceToHost);
        if (FILE* f = fopen(profPath, "w")) {
            fprintf(f, "task,I,J,level,nterms,t_claim,t_terms,t_deps,t_end\n");
            for (int t = 0; t < sym.nTasks; ++t)
                fprintf(f, "%d,%d,%d,%d,%lld,%llu,%llu,%llu,%llu\n", t, sym.taskI[t], sym.taskJ[t], sym.level[sym.taskJ[t]],
                        (long long)(sym.termPtr[t + 1] - sym.termPtr[t]), hp[4 * t] - hp[0], hp[4 * t + 1] - hp[0], hp[4 * t + 2] - hp[0], hp[4 * t + 3] - hp[0]);
            fclose(f);
        }
        cudaFree(dprof);
    }
    cudaEventDestroy(e2);
    (void)bestF;
    int info = 0; double mn = 0, mx = 0;
    tchol_pivot_stats(tc, &info, &mn, &mx, st);
    std::vector<double> hx(sym.ld);
    cudaMemcpy(hx.data(), tc.xs, sizeof(double) * sym.ld, cudaMemcpyDeviceToHost);
    for (int64_t c = 0; c < n; ++c) x[c] = hx[x2s[c]];
    if (stats) {
        stats[0] = best; stats[1] = sym.nT; stats[2] = sym.nSlots; stats[3] = sym.nTasks; stats[4] = (double)sym.nTerms;
        stats[5] = sym.depth; stats[6] = mn; stats[7] = mx;
    }
    cudaError_t e = cudaDeviceSynchronize();
    tchol_free(tc); cudaFree(d0); cudaFree(drhs);
    cudaEventDestroy(e0); cudaEventDestroy(e1); cudaStreamDestroy(st);
    if (e != cudaSuccess) { g_create_err = std::string("dbat_tile_chol_solve: ") + cudaGetErrorString(e); return DBAT_E_CUDA; }
    return info != 0 ? DBAT_E_NOTSPD : DBAT_OK;
}

// --------------------------------------------------------------------------------------------
// dbat_set_devices: one process, several devices (SURVEY §8b: a MATLAB mexFunction has one interpreter thread,
// code/test/postcov/icpc_mex.c:495, and cannot be launched once per GPU).  The handle becomes the front of a group:
// the object points are cut into one range per device, every device gets its own sub-problem (created from the
// retained copy of the description) on its own persistent host thread, the sub-problems are joined by NCCL exactly
// like the ranks of a multi-process run, and every API call on the front handle runs on all of them and merges the
// results (camera part from the first device, every point and observation from its owner).
// --------------------------------------------------------------------------------------------
struct DescCopy {
    dbat_problem_desc d;
    std::vector<double> IOval, EOval, OPval, IPval, IPstd, pxSize, prior_val, prior_std;
    std::vector<int64_t> IPimg, IPop, IOs, IOd, EOs, EOd, OPs, OPd, prior_x, ca, cb;
    void bind() {
        d.IOval = IOval.data(); d.EOval = EOval.data(); d.OPval = OPval.data(); d.IPval = IPval.data(); d.IPstd = IPstd.data();
        d.IPimg = IPimg.data(); d.IPop = IPop.data(); d.pxSize = pxSize.data();
        d.IOdes_src = IOs.data(); d.IOdes_dest = IOd.data(); d.EOdes_src = EOs.data(); d.EOdes_dest = EOd.data();
        d.OPdes_src = OPs.data(); d.OPdes_dest = OPd.data();
        d.prior_x = prior_x.data(); d.prior_val = prior_val.data(); d.prior_std = prior_std.data();
        d.covis_a = ca.data(); d.covis_b = cb.data(); d.nCovis = (int64_t)ca.size();
    }
};
static DescCopy* copy_desc(const dbat_problem_desc* d, int NC) {
    DescCopy* c = new DescCopy();
    c->d = *d;
    const size_t nImg = (size_t)d->nImg, nOP = (size_t)d->nOP, nIP = (size_t)d->nIP;
    const size_t nPr = (size_t)(d->nPriorIO + d->nPriorEO + d->nPriorOP);
    c->IOval.assign(d->IOval, d->IOval + (size_t)NC * nImg); c->EOval.assign(d->EOval, d->EOval + 6 * nImg);
    c->OPval.assign(d->OPval, d->OPval + 3 * nOP); c->IPval.assign(d->IPval, d->IPval + 2 * nIP);
    c->IPstd.assign(d->IPstd, d->IPstd + 2 * nIP); c->pxSize.assign(d->pxSize, d->pxSize + 2 * nImg);
    c->IPimg.assign(d->IPimg, d->IPimg + nIP); c->IPop.assign(d->IPop, d->IPop + nIP);
    c->IOs.assign(d->IOdes_src, d->IOdes_src + d->nIOdes); c->IOd.assign(d->IOdes_dest, d->IOdes_dest + d->nIOdes);
    c->EOs.assign(d->EOdes_src, d->EOdes_src + d->nEOdes); c->EOd.assign(d->EOdes_dest, d->EOdes_dest + d->nEOdes);
    c->OPs.assign(d->OPdes_src, d->OPdes_src + d->nOPdes); c->OPd.assign(d->OPdes_dest, d->OPdes_dest + d->nOPdes);
    if (nPr) { c->prior_x.assign(d->prior_x, d->prior_x + nPr); c->prior_val.assign(d->prior_val, d->prior_val + nPr); c->prior_std.assign(d->prior_std, d->prior_std + nPr); }
    if (d->nCovis > 0 && d->covis_a && d->covis_b) { c->ca.assign(d->covis_a, d->covis_a + d->nCovis); c->cb.assign(d->covis_b, d->covis_b + d->nCovis); }
    c->bind();
    return c;
}
static void free_desc(DescCopy* c) { delete c; }

struct GroupWorker {
    std::thread th; std::mutex m; std::condition_variable cv;
    std::function<void()> job; bool has = false, quit = false;
};
struct DevGroup {
    int ndev = 0;
    std::vector<int> dev;
    std::vector<dbat_handle*> sub;
    std::vector<std::unique_ptr<GroupWorker>> w;
    std::vector<int> lo, hi;                         // object-point range of every device
    std::vector<std::vector<int64_t>> obs;           // per device: global observation index of its observations
    std::vector<std::vector<int64_t>> prow;          // per device: global prior-row index of its prior rows
    std::vector<std::vector<int64_t>> ownCols;       // per device: x columns of its object points (0-based)
    std::vector<std::unique_ptr<DescCopy>> sd;
    int nC = 0;
    void run_all(const std::function<void(int)>& fn) {
        std::mutex dm; std::condition_variable dcv; int left = ndev;
        for (int r = 0; r < ndev; ++r) {
            GroupWorker& k = *w[r];
            std::lock_guard<std::mutex> g(k.m);
            k.job = [&, r]() { fn(r); { std::lock_guard<std::mutex> g2(dm); --left; } dcv.notify_one(); };
            k.has = true;
            k.cv.notify_one();
        }
        std::unique_lock<std::mutex> lk(dm);
        dcv.wait(lk, [&] { return left == 0; });
    }
};
static void worker_loop(GroupWorker* k, int device) {
    cudaSetDevice(device);
    for (;;) {
        std::function<void()> job;
        {
            std::unique_lock<std::mutex> lk(k->m);
            k->cv.wait(lk, [&] { return k->has || k->quit; });
            if (k->quit && !k->has) return;
            job.swap(k->job); k->has = false;
        }
        job();
    }
}
static const dbat_handle* group_first(const dbat_handle* h) { return h->group->sub[0]; }
static void group_destroy(dbat_handle* h) {
    DevGroup* G = h->group;
    G->run_all([&](int r) { if (G->sub[r]) { dbat_destroy(G->sub[r]); G->sub[r] = nullptr; } });
    for (auto& k : G->w) { { std::lock_guard<std::mutex> g(k->m); k->quit = true; } k->cv.notify_one(); k->th.join(); }
    delete G;
    h->group = nullptr;
}

extern "C" int dbat_set_devices(dbat_handle* h, const int* dev, int ndev) {
    if (!h || !dev || ndev < 1) return DBAT_E_BADARG;
    if (h->group) { h->err = "dbat_set_devices was already called on this handle"; return DBAT_E_STATE; }
    if (h->nranks > 1) { h->err = "the handle is a rank of a multi-process run"; return DBAT_E_STATE; }
    if (!h->dcopy) { h->err = "no description retained"; return DBAT_E_STATE; }
    int have = 0;
    cudaGetDeviceCount(&have);
    for (int r = 0; r < ndev; ++r) if (dev[r] < 0 || dev[r] >= have) { h->err = "device index out of range"; return DBAT_E_BADARG; }
    const dbat_problem_desc& D = h->dcopy->d;
    const int nOP = (int)D.nOP, nImg = (int)D.nImg, nObs = (int)D.nIP;
    DevGroup* G = new DevGroup();
    G->ndev = ndev; G->dev.assign(dev, dev + ndev); G->sub.assign(ndev, nullptr); G->nC = h->P.nC;
    // contiguous point ranges balanced by observation count (parallel.py:partition_points)
    {
        std::vector<int64_t> cum((size_t)nOP + 1, 0);
        for (int k = 0; k < nObs; ++k) cum[(size_t)D.IPop[k]]++;
        for (int j = 0; j < nOP; ++j) cum[(size_t)j + 1] += cum[(size_t)j];
        G->lo.assign(ndev, 0); G->hi.assign(ndev, nOP);
        for (int r = 1; r < ndev; ++r) {
            const int64_t target = cum[(size_t)nOP] * r / ndev;
            int b = (int)(std::lower_bound(cum.begin(), cum.end(), target) - cum.begin());
            b = std::max(G->lo[r - 1], std::min(b, nOP));
            G->lo[r] = b; G->hi[r - 1] = b;
        }
    }
    // global co-visibility edges (the front handle analysed the whole project at create)
    std::vector<int64_t> ea, eb;
    for (int i = 0; i < nImg; ++i)
        for (int64_t k = h->plan.adjPtr[i]; k < h->plan.adjPtr[i + 1]; ++k) if (h->plan.adj[k] > i) { ea.push_back(i + 1); eb.push_back(h->plan.adj[k] + 1); }
    G->obs.resize(ndev); G->prow.resize(ndev); G->ownCols.resize(ndev); G->sd.resize(ndev);
    const int64_t nPr = D.nPriorIO + D.nPriorEO + D.nPriorOP;
    for (int r = 0; r < ndev; ++r) {
        const int lo = G->lo[r], hi = G->hi[r];
        std::unique_ptr<DescCopy> c(new DescCopy());
        const DescCopy& A = *h->dcopy;
        c->d = A.d;
        c->IOval = A.IOval; c->EOval = A.EOval; c->pxSize = A.pxSize;
        c->IOs = A.IOs; c->IOd = A.IOd; c->EOs = A.EOs; c->EOd = A.EOd;
        c->OPval.assign(A.OPval.begin() + 3 * (size_t)lo, A.OPval.begin() + 3 * (size_t)hi);
        for (int k = 0; k < nObs; ++k) {
            const int64_t j = A.IPop[k] - 1;
            if (j < lo || j >= hi) continue;
            G->obs[r].push_back(k);
            c->IPimg.push_back(A.IPimg[k]); c->IPop.push_back(j - lo + 1);
            c->IPval.push_back(A.IPval[2 * (size_t)k]); c->IPval.push_back(A.IPval[2 * (size_t)k + 1]);
            c->IPstd.push_back(A.IPstd[2 * (size_t)k]); c->IPstd.push_back(A.IPstd[2 * (size_t)k + 1]);
        }
        std::vector<char> own((size_t)D.n, 0);
        for (int64_t k = 0; k < D.nOPdes; ++k) {
            const int64_t dd = A.OPd[k] - 1;
            if (dd < 3 * (int64_t)lo || dd >= 3 * (int64_t)hi) continue;
            c->OPs.push_back(A.OPs[k]); c->OPd.push_back(dd - 3 * (int64_t)lo + 1);
            own[(size_t)(A.OPs[k] - 1)] = 1; G->ownCols[r].push_back(A.OPs[k] - 1);
        }
        int64_t nIO = 0, nEO = 0, nOPp = 0;
        for (int64_t q = 0; q < nPr; ++q) {
            const bool isCam = q < D.nPriorIO + D.nPriorEO;
            if (isCam ? (r != 0) : !own[(size_t)(A.prior_x[q] - 1)]) continue;
            c->prior_x.push_back(A.prior_x[q]); c->prior_val.push_back(A.prior_val[q]); c->prior_std.push_back(A.prior_std[q]);
            G->prow[r].push_back(q);
            if (q < D.nPriorIO) ++nIO; else if (isCam) ++nEO; else ++nOPp;
        }
        c->ca = ea; c->cb = eb;
        c->d.nOP = hi - lo; c->d.nIP = (int64_t)G->obs[r].size();
        c->d.nOPdes = (int64_t)c->OPs.size();
        c->d.nPriorIO = nIO; c->d.nPriorEO = nEO; c->d.nPriorOP = nOPp;
        c->bind();
        G->sd[r] = std::move(c);
    }
    for (int r = 0; r < ndev; ++r) {
        G->w.emplace_back(new GroupWorker());
        G->w[r]->th = std::thread(worker_loop, G->w[r].get(), dev[r]);
    }
    std::vector<int> rcs(ndev, 0);
    std::vector<std::string> errs(ndev);
    G->run_all([&](int r) {
        g_in_group_create = true;
        rcs[r] = dbat_create(&G->sd[r]->d, &G->sub[r]);
        g_in_group_create = false;
        if (rcs[r]) errs[r] = g_create_err;
    });
    int rc = 0;
    for (int r = 0; r < ndev; ++r) if (rcs[r]) { rc = rcs[r]; h->err = "device " + std::to_string(dev[r]) + ": " + errs[r]; }
    if (!rc && ndev > 1) {
        char uid[128];
        rc = dbat_comm_unique_id(uid);
        if (rc) h->err = "ncclGetUniqueId failed";
        if (!rc) {
            G->run_all([&](int r) { rcs[r] = dbat_comm_init(G->sub[r], ndev, r, uid); if (rcs[r]) errs[r] = G->sub[r]->err; });
            for (int r = 0; r < ndev; ++r) if (rcs[r]) { rc = rcs[r]; h->err = "device " + std::to_string(dev[r]) + ": " + errs[r]; }
        }
    }
    h->group = G;
    if (rc) { group_destroy(h); return rc; }
    for (auto& c : G->sd) c.reset();                  // the sub-problems hold their own copies now
    return DBAT_OK;
}

static int group_rc(dbat_handle* h, const std::vector<int>& rcs) {
    DevGroup* G = h->group;
    for (int r = 0; r < G->ndev; ++r)
        if (rcs[r]) { h->err = "device " + std::to_string(G->dev[r]) + ": " + G->sub[r]->err; return rcs[r]; }
    return DBAT_OK;
}
static void group_merge_x(DevGroup* G, int n, const std::vector<std::vector<double>>& part, double* out) {
    // camera part from the first device, every point column from its owner; columns nobody owns (none) keep part[0]
    memcpy(out, part[0].data(), sizeof(double) * (size_t)n);
    for (int r = 1; r < G->ndev; ++r) for (int64_t c : G->ownCols[r]) out[c] = part[r][(size_t)c];
}
static void group_merge_r(dbat_handle* h, const std::vector<std::vector<double>>& part, double* out) {
    DevGroup* G = h->group;
    const int64_t nObs = h->P.nObs;
    for (int r = 0; r < G->ndev; ++r) {
        const std::vector<int64_t>& ob = G->obs[r];
        for (size_t k = 0; k < ob.size(); ++k) { out[2 * ob[k]] = part[r][2 * k]; out[2 * ob[k] + 1] = part[r][2 * k + 1]; }
        for (size_t q = 0; q < G->prow[r].size(); ++q) out[2 * nObs + G->prow[r][q]] = part[r][2 * ob.size() + q];
    }
}
static int group_eval(dbat_handle* h, const double* x, double* r, int weighted) {
    DevGroup* G = h->group;
    std::vector<int> rcs(G->ndev, 0);
    std::vector<std::vector<double>> part(G->ndev);
    G->run_all([&](int k) {
        part[k].resize((size_t)std::max<int64_t>(1, dbat_num_residuals(G->sub[k])));
        rcs[k] = dbat_eval(G->sub[k], x, r ? part[k].data() : nullptr, weighted);
    });
    int rc = group_rc(h, rcs);
    if (!rc && r) group_merge_r(h, part, r);
    return rc;
}
static int group_normal_step(dbat_handle* h, const double* x, double lambda, int flags, double* p, double* stats) {
    DevGroup* G = h->group;
    const int n = h->P.n;
    std::vector<int> rcs(G->ndev, 0);
    std::vector<std::vector<double>> part(G->ndev), st(G->ndev, std::vector<double>(8, 0.0));
    G->run_all([&](int k) {
        if (p) part[k].assign((size_t)n, 0.0);
        rcs[k] = dbat_normal_step(G->sub[k], x, lambda, flags, p ? part[k].data() : nullptr, st[k].data());
    });
    int rc = group_rc(h, rcs);
    if (rc) return rc;
    if (p) group_merge_x(G, n, part, p);
    if (stats) { memcpy(stats, st[0].data(), sizeof(double) * 8); for (int k = 1; k < G->ndev; ++k) stats[6] = std::max(stats[6], st[k][6]); }
    return DBAT_OK;
}
static int group_solve(dbat_handle* h, int method, const dbat_opts* opts, const double* x0, dbat_result* res) {
    DevGroup* G = h->group;
    const int n = h->P.n, cap = opts->maxIter + 2;
    struct Buf { std::vector<double> x, p, rw, ru, tr, rr, dmp, rho; std::vector<int32_t> steps; dbat_result r; };
    std::vector<Buf> B(G->ndev);
    std::vector<int> rcs(G->ndev, 0);
    G->run_all([&](int k) {
        Buf& b = B[k];
        const size_t mk = (size_t)std::max<int64_t>(1, dbat_num_residuals(G->sub[k]));
        b.x.assign(n, 0.0); b.p.assign(n, 0.0); b.rr.assign(cap + 1, NAN); b.dmp.assign(cap + 1, NAN); b.rho.assign(cap, NAN); b.steps.assign(cap, 0);
        memset(&b.r, 0, sizeof(b.r));
        b.r.x = b.x.data(); b.r.p = res->p ? b.p.data() : nullptr;
        if (res->r_w) { b.rw.assign(mk, 0.0); b.r.r_w = b.rw.data(); }
        if (res->r_u) { b.ru.assign(mk, 0.0); b.r.r_u = b.ru.data(); }
        if (res->trace) { b.tr.assign((size_t)n * cap, NAN); b.r.trace = b.tr.data(); }
        b.r.rr = b.rr.data(); b.r.damping = b.dmp.data(); b.r.rhos = res->rhos ? b.rho.data() : nullptr; b.r.steps = res->steps ? b.steps.data() : nullptr;
        rcs[k] = dbat_solve(G->sub[k], method, opts, x0, &b.r);
    });
    int rc = group_rc(h, rcs);
    if (rc) return rc;
    const dbat_result& r0 = B[0].r;
    res->code = r0.code; res->iters = r0.iters; res->nTrace = r0.nTrace; res->nRr = r0.nRr; res->nDamping = r0.nDamping; res->nRhos = r0.nRhos;
    res->seconds = r0.seconds; res->launches = r0.launches;
    memcpy(res->rr, B[0].rr.data(), sizeof(double) * (cap + 1));
    memcpy(res->damping, B[0].dmp.data(), sizeof(double) * (cap + 1));
    if (res->rhos) memcpy(res->rhos, B[0].rho.data(), sizeof(double) * cap);
    if (res->steps) memcpy(res->steps, B[0].steps.data(), sizeof(int32_t) * cap);
    std::vector<std::vector<double>> part(G->ndev);
    for (int k = 0; k < G->ndev; ++k) part[k].swap(B[k].x);
    group_merge_x(G, n, part, res->x);
    if (res->p) { for (int k = 0; k < G->ndev; ++k) part[k].swap(B[k].p); group_merge_x(G, n, part, res->p); }
    if (res->r_w) { for (int k = 0; k < G->ndev; ++k) part[k].swap(B[k].rw); group_merge_r(h, part, res->r_w); }
    if (res->r_u) { for (int k = 0; k < G->ndev; ++k) part[k].swap(B[k].ru); group_merge_r(h, part, res->r_u); }
    if (res->trace)
        for (int c = 0; c < std::min(res->nTrace, cap); ++c) {
            memcpy(res->trace + (size_t)c * n, B[0].tr.data() + (size_t)c * n, sizeof(double) * (size_t)n);
            for (int k = 1; k < G->ndev; ++k) for (int64_t col : G->ownCols[k]) res->trace[(size_t)c * n + col] = B[k].tr[(size_t)c * n + col];
        }
    return DBAT_OK;
}
static int group_cov(dbat_handle* h, int which, double s0, double* out) {
    DevGroup* G = h->group;
    if (which == DBAT_COV_CXX || which == DBAT_COV_CXX_OP) { h->err = "the dense point covariance is single-device only; use COP"; return DBAT_E_UNSUPPORTED; }
    std::vector<int> rcs(G->ndev, 0);
    std::vector<std::vector<double>> part(G->ndev);
    const size_t camSize = which == DBAT_COV_CIO ? (size_t)h->plan.NC * h->plan.NC * h->P.nImg : which == DBAT_COV_CEO ? (size_t)36 * h->P.nImg : (size_t)G->nC * G->nC;
    G->run_all([&](int k) {
        part[k].assign(which == DBAT_COV_COP ? (size_t)9 * std::max(1, G->hi[k] - G->lo[k]) : std::max<size_t>(1, camSize), 0.0);
        rcs[k] = dbat_cov(G->sub[k], which, s0, part[k].data());
    });
    bool notspd = false;
    for (int k = 0; k < G->ndev; ++k) if (rcs[k] == DBAT_E_NOTSPD) { notspd = true; rcs[k] = 0; }
    int rc = group_rc(h, rcs);
    if (rc) return rc;
    if (which == DBAT_COV_COP) { for (int k = 0; k < G->ndev; ++k) memcpy(out + 9 * (size_t)G->lo[k], part[k].data(), sizeof(double) * 9 * (size_t)(G->hi[k] - G->lo[k])); }
    else memcpy(out, part[0].data(), sizeof(double) * camSize);
    return notspd ? DBAT_E_NOTSPD : DBAT_OK;
}

// --------------------------------------------------------------------------------------------
// multi-GPU plumbing
// --------------------------------------------------------------------------------------------
extern "C" int dbat_comm_unique_id(void* id128) {
    if (!id128) return DBAT_E_BADARG;
    if (!nccl_load()) { g_create_err = "libnccl.so.2 not found"; return DBAT_E_NCCL; }
    nccl_uid id;
    if (g_nccl.GetUniqueId(&id) != 0) return DBAT_E_NCCL;
    memcpy(id128, &id, sizeof(id));
    return DBAT_OK;
}
extern "C" int dbat_comm_init(dbat_handle* h, int nranks, int rank, const void* id128) {
    if (!h || !id128 || nranks < 1 || rank < 0 || rank >= nranks) return DBAT_E_BADARG;
    if (nranks == 1) { h->nranks = 1; h->rank = 0; return DBAT_OK; }
    if (!nccl_load()) { h->err = "libnccl.so.2 not found"; return DBAT_E_NCCL; }
    nccl_uid id; memcpy(&id, id128, sizeof(id));
    int rc = g_nccl.CommInitRank(&h->comm, nranks, id, rank);
    if (rc != 0) { h->err = std::string("ncclCommInitRank: ") + (g_nccl.GetErrorString ? g_nccl.GetErrorString(rc) : "?"); return DBAT_E_NCCL; }
    h->nranks = nranks; h->rank = rank;
    // distribute the factorisation: cut the elimination tree into one subtree per rank (tilesym.cu)
    TileSym sym;
    if ((rc = analyse_reduced(h, nranks, rank, sym))) return rc;
    // the window Schur index was built at create for the one-part order: its camera-pair blocks are lower
    // triangular in S only while the images with columns in S keep that order
    if (!plan_same_order(h->plan, h->tc.sym, sym)) {
        h->err = "the distributed elimination order differs from the one the window Schur index was built for";
        return DBAT_E_STATE;
    }
    return setup_reduced(h, sym);
}
