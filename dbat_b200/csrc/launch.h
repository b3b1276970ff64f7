// launch.h — host-side launchers (one per kernel family) shared by the translation units.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

struct DevProblem;

// every kernel launch of the library is counted (reported as gpu_launches by bench.py)
extern int64_t g_dbat_launches;
static inline void count_launch(int n = 1) { __atomic_fetch_add(&g_dbat_launches, (int64_t)n, __ATOMIC_RELAXED); }

// eval.cu
struct ScatterList { const int* src; const int* dest; double* arr; int cnt; int nb; };
void launch_set_params(const DevProblem& P, const double* x, ScatterList io, ScatterList eo, ScatterList op,
                       const int* rep, int nIO, cudaStream_t st);
void launch_cam_side(const DevProblem& P, const int* img_chunk_start, double* tmp, cudaStream_t st);
void launch_point_side(const DevProblem& P, cudaStream_t st);
void launch_prior_apply(const DevProblem& P, const double* x, double* camDiag, double* camG,
                        const int* col2pt, bool clear, cudaStream_t st);
void launch_resid(const DevProblem& P, const double* x, double* partial, double* scal, int slot,
                  double* r_out, int weighted, cudaStream_t st);
void launch_prior_rr(const DevProblem& P, const double* x, double* partial, double* scal, int slot, bool clear, cudaStream_t st);
void launch_jp(const DevProblem& P, const double* x, const double* p, double* partial, double* scal,
               int slot2, int slotr, cudaStream_t st);
void launch_export_jac(const DevProblem& P, double* out, int weighted, cudaStream_t st);
void launch_export_mask(const DevProblem& P, unsigned long long* out, cudaStream_t st);

// schur.cu
void launch_diag(const DevProblem& P, const double* camDiag, double* diagN, cudaStream_t st);
void launch_build_S(const DevProblem& P, const double* camDiag, const double* camG, double lambda,
                    cudaStream_t st);
void launch_schur(const DevProblem& P, double lambda, cudaStream_t st);
void launch_point_vinv(const DevProblem& P, double lambda, cudaStream_t st);   // P.vinv = (V_j + lambda I)^-1
void launch_scale_prep(const DevProblem& P, const double* d, double* dS, cudaStream_t st);
void launch_unpermute(const DevProblem& P, const double* xs, const double* d, double* pc, double* pEO, cudaStream_t st);
void launch_backsub(const DevProblem& P, double lambda, const double* pc, const double* pEO, double* p, double* partial,
                    const double* camDiag, const double* camG, double* jpOut, cudaStream_t st,
                    cudaStream_t st2 = nullptr, cudaEvent_t evFork = nullptr, cudaEvent_t evJoin = nullptr);
void launch_vec_ops_sum(const double* a, int n, double* partial, double* scal, int slot, cudaStream_t st);
void launch_dot(const double* a, const double* b, int n, double* partial, double* scal, int slot, cudaStream_t st);
void launch_axpy(double alpha, const double* x, const double* y, double* out, int n, cudaStream_t st);
void launch_inv_sqrt(const double* in, double* out, int n, cudaStream_t st);
void launch_mul(const double* a, const double* b, double* out, int n, cudaStream_t st);

// schur_win.cu (Schur reduction: window accumulation per point cluster + fixed-order sums, no atomics)
void launch_schur_win(const DevProblem& P, double lambda, const double* shAcc, cudaStream_t st);

// general_io.cu (general IO block structure)
void launch_point_side_gen(const DevProblem& P, cudaStream_t st);
void launch_build_S_gen(const DevProblem& P, const double* camDiag, const double* camG, double lambda, cudaStream_t st);
void launch_schur_gen(const DevProblem& P, double lambda, cudaStream_t st);
int launch_backsub_gen(const DevProblem& P, double lambda, double* p, double* stats, cudaStream_t st);
void launch_cop_gen(const DevProblem& P, const double* C, int ldc, const double* dsc, double s02, double* out, cudaStream_t st);
void launch_io_diag_grad_gen(const DevProblem& P, const double* camDiag, const double* camG, double* diagN, double* grad,
                             cudaStream_t st);

// chol.cu
struct CholWork {
    int ld = 0, nb = 0;             // leading dimension (multiple of 128), # 128-blocks
    double* invL = nullptr;         // nb x 128 x 128 inverses of the diagonal blocks
    int* info = nullptr;            // device flag: 0 ok, k > 0: block k - 1 holds the first non-positive pivot
};
int chol_alloc(CholWork& w, int ld);          // 0 ok, 1 out of memory (nothing left allocated)
void chol_free(CholWork& w);
// In-place lower Cholesky of the ld x ld column-major matrix A (rows/cols past the order of the
// matrix are padding and must hold the identity).  Asynchronous; read w.info afterwards.
void chol_factor(const CholWork& w, double* A, cudaStream_t st);
// After chol_factor: Z (ld x ld) = inv(L)', C (ld x ld) = inv(A), full symmetric.
void chol_inverse(const CholWork& w, const double* A, double* Z, double* C, cudaStream_t st);
