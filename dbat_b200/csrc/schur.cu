// schur.cu — damped step: batched 3x3 point-block inverses, Schur reduction onto the dense
// camera/IO system, back-substitution.  Replaces `p=(JTJ+lambda*I)\(-JTr)`
// (code/bundle/lsa/levenberg_marquardt.m:119) and the Jacobi-scaled variant
// (gauss_newton_armijo.m:166-174) with the block elimination of SURVEY.md Appendix A:
//   S = N_cc + lambda*I - sum_j W~_j (V_j + lambda*I)^-1 W~_j',   rhs = -g_c + sum_j W~_j (..)^-1 g_j
//   p_j = (V_j + lambda*I)^-1 (-g_j - W~_j' p_c)
#include "kernels.cuh"
#include <algorithm>
#include "launch.h"

__device__ __forceinline__ double gram_at(const double* __restrict__ G, int R, int C) {
    if (R < C) { const int t = R; R = C; C = t; }
    const int p = R >> 3, q = C >> 3, i = R & 7, j = C & 7;
    const int tp = p * (p + 1) / 2 + q;
    return G[tp * 64 + (i * 4 + (j >> 1)) * 2 + (j & 1)];
}

// inverse of the damped 3x3 point block; fixed coordinates (mask 0) get a unit diagonal.
// Cholesky based (the block is SPD).  Returns false if not positive definite.
__device__ __forceinline__ bool point_inverse(const double* __restrict__ rec, const int* __restrict__ opc,
                                              double lambda, double Vi[6]) {
    double a00 = rec[0], a01 = rec[1], a02 = rec[2], a11 = rec[3], a12 = rec[4], a22 = rec[5];
    const bool f0 = opc[0] >= 0, f1 = opc[1] >= 0, f2 = opc[2] >= 0;
    a00 = f0 ? a00 + lambda : 1.0;
    a11 = f1 ? a11 + lambda : 1.0;
    a22 = f2 ? a22 + lambda : 1.0;
    bool ok = a00 > 0.0;
    const double l00 = sqrt(a00);
    const double l10 = a01 / l00, l20 = a02 / l00;
    const double d1 = a11 - l10 * l10;
    ok = ok && d1 > 0.0;
    const double l11 = sqrt(d1);
    const double l21 = (a12 - l20 * l10) / l11;
    const double d2 = a22 - l20 * l20 - l21 * l21;
    ok = ok && d2 > 0.0;
    const double l22 = sqrt(d2);
    // M = inv(L)
    const double m00 = 1.0 / l00, m11 = 1.0 / l11, m22 = 1.0 / l22;
    const double m10 = -l10 * m00 * m11;
    const double m21 = -l21 * m11 * m22;
    const double m20 = -(l20 * m00 + l21 * m10) * m22;
    // Vi = M' M
    Vi[0] = m00 * m00 + m10 * m10 + m20 * m20;
    Vi[1] = m10 * m11 + m20 * m21;
    Vi[2] = m20 * m22;
    Vi[3] = m11 * m11 + m21 * m21;
    Vi[4] = m21 * m22;
    Vi[5] = m22 * m22;
    if (!f0) { Vi[0] = 0.0; Vi[1] = 0.0; Vi[2] = 0.0; }
    if (!f1) { Vi[1] = 0.0; Vi[3] = 0.0; Vi[4] = 0.0; }
    if (!f2) { Vi[2] = 0.0; Vi[4] = 0.0; Vi[5] = 0.0; }
    return ok;
}

__device__ __forceinline__ void symv3(const double Vi[6], const double w[3], double y[3]) {
    y[0] = Vi[0] * w[0] + Vi[1] * w[1] + Vi[2] * w[2];
    y[1] = Vi[1] * w[0] + Vi[3] * w[1] + Vi[4] * w[2];
    y[2] = Vi[2] * w[0] + Vi[4] * w[1] + Vi[5] * w[2];
}

// diag(J'J) for every unknown (Jacobi scaling, trace for lambda0)
__global__ void k_diag(DevProblem P, const double* __restrict__ camDiag, double* __restrict__ diagN) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < DBAT_NSLOT) {
        const int c = P.sh_col[t];
        if (c >= 0) diagN[c] = gram_at(P.shG, t, t) + camDiag[c];
    }
    if (t < P.nImg * 6) {
        const int i = t / 6, a = t % 6;
        const int c = P.eo_col[t];
        if (c >= 0) diagN[c] = gram_at(P.imgG + (size_t)i * DBAT_GSZ, DBAT_COL_EO + a, DBAT_COL_EO + a) + camDiag[c];
    }
    if (t < P.nOP * 3) {
        const int j = t / 3, a = t % 3;
        const int c = P.op_col[t];
        if (c >= 0) diagN[c] = P.pt[(size_t)j * DBAT_PT_STRIDE + (a == 0 ? 0 : (a == 1 ? 3 : 5))];
    }
}
void launch_diag(const DevProblem& P, const double* camDiag, double* diagN, cudaStream_t st) {
    if (P.ioGeneral) {      // IO columns: prior term, then the Gram diagonals of every image that uses the column
        cudaMemcpyAsync(diagN, camDiag, sizeof(double) * P.nC, cudaMemcpyDeviceToDevice, st);
        launch_io_diag_grad_gen(P, camDiag, nullptr, diagN, nullptr, st);
    }
    int n = P.nOP * 3;
    if (P.nImg * 6 > n) n = P.nImg * 6;
    if (DBAT_NSLOT > n) n = DBAT_NSLOT;
    k_diag<<<(n + 255) / 256, 256, 0, st>>>(P, camDiag, diagN);
    count_launch();
}

// S := N_cc + lambda*I (lower triangle, S order), rhs := -g_c ; padding positions get a unit diagonal
__global__ void k_build_S(DevProblem P, const double* __restrict__ camDiag, const double* __restrict__ camG,
                          double lambda) {
    const int i = blockIdx.x;         // image index, or nImg for the shared block
    if (i < P.nImg) {
        const double* G = P.imgG + (size_t)i * DBAT_GSZ;
        const int* ec = P.eo_col + 6 * (size_t)i;
        const int* es = P.eo_s + 6 * (size_t)i;
        for (int e = threadIdx.x; e < 6 * (6 + DBAT_NSLOT + 1); e += blockDim.x) {
            const int a = e / (6 + DBAT_NSLOT + 1), b = e % (6 + DBAT_NSLOT + 1);
            const int row = es[a];
            if (row < 0) continue;
            if (b < 6) {                                   // EO x EO (S indices ascend with the element)
                const int col = es[b];
                if (col < 0 || col > row) continue;
                double v = gram_at(G, DBAT_COL_EO + a, DBAT_COL_EO + b);
                if (a == b) v += camDiag[ec[a]] + lambda;
                *tc_at(P.T, row, col) = v;
            } else if (b < 6 + DBAT_NSLOT) {               // shared IO x EO (the IO block comes last in S)
                const int srow = P.sh_s[b - 6];
                if (srow < 0) continue;
                *tc_at(P.T, srow, row) = gram_at(G, DBAT_COL_EO + a, b - 6);
            } else {
                P.rhs[row] = -(gram_at(G, DBAT_COL_EO + a, DBAT_COL_R) + camG[ec[a]]);
            }
        }
    } else if (i == P.nImg) {
        for (int e = threadIdx.x; e < DBAT_NSLOT * (DBAT_NSLOT + 1); e += blockDim.x) {
            const int a = e / (DBAT_NSLOT + 1), b = e % (DBAT_NSLOT + 1);
            const int row = P.sh_s[a];
            if (row < 0) continue;
            if (b < DBAT_NSLOT) {
                const int col = P.sh_s[b];
                if (col < 0 || col > row) continue;
                double v = gram_at(P.shG, a, b);
                if (a == b) v += camDiag[P.sh_col[a]] + lambda;
                *tc_at(P.T, row, col) = v;
            } else {
                P.rhs[row] = -(gram_at(P.shG, a, DBAT_COL_R) + camG[P.sh_col[a]]);
            }
        }
    }
    // padding positions: one thread each, spread over all blocks (a single block walking ldS entries cost 28 us)
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k < P.ldS && P.s2x[k] < 0) {
        P.rhs[k] = 0.0;
        if (k != P.ldS - 1) *tc_at(P.T, k, k) = 1.0;         // the rhs row gets its diagonal in tchol_put_rhs
    }
}
void launch_build_S(const DevProblem& P, const double* camDiag, const double* camG, double lambda,
                    cudaStream_t st) {
    if (P.ioGeneral) { launch_build_S_gen(P, camDiag, camG, lambda, st); return; }
    tchol_zero_dev(P.T, st);
    k_build_S<<<std::max(P.nImg + 1, (P.ldS + 127) / 128), 128, 0, st>>>(P, camDiag, camG, lambda);
    count_launch();
}

// (V_j + lambda I)^-1 of every point into P.vinv (the point blocks of the covariance, dbat_cov)
__global__ void k_point_vinv(DevProblem P, double lambda) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= P.nOP) return;
    double Vi[6];
    point_inverse(P.pt + (size_t)j * DBAT_PT_STRIDE, P.op_col + 3 * (size_t)j, lambda, Vi);
    double2* o = reinterpret_cast<double2*>(P.vinv + (size_t)j * 8);
    o[0] = make_double2(Vi[0], Vi[1]); o[1] = make_double2(Vi[2], Vi[3]); o[2] = make_double2(Vi[4], Vi[5]);
}

void launch_point_vinv(const DevProblem& P, double lambda, cudaStream_t st) {
    if (P.nOP > 0) { k_point_vinv<<<(P.nOP + 255) / 256, 256, 0, st>>>(P, lambda); count_launch(); }
}
void launch_schur(const DevProblem& P, double lambda, cudaStream_t st) {
    if (P.nOP <= 0) return;
    if (P.ioGeneral) { launch_schur_gen(P, lambda, st); return; }
    // the wide points (more than DBAT_GRP_MAXM rays; none at BASELINE configs 4 / 5) first (schur_wide.cu), then the
    // window accumulation + fixed-order reduction of all others (schur_win.cu), which adds the wide points' shared x
    // shared table; every step of both is in a fixed order
    const double* shAcc = nullptr;
    if (P.nBig > 0) {
        launch_schur_wide(P, lambda, st);
        shAcc = P.wide_shAcc;
    }
    launch_schur_win(P, lambda, shAcc, st);
}

// Jacobi column scaling (gauss_newton_armijo.m:166-172) of the reduced system: dS[s] = d[x column of s]
// (1 at padding positions), rhs := D rhs; the tiles are scaled by tchol_scale.
__global__ void k_scale_prep(DevProblem P, const double* __restrict__ d, double* __restrict__ dS) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= P.ldS) return;
    const int c = P.s2x[s];
    const double v = c >= 0 ? d[c] : 1.0;
    dS[s] = v;
    P.rhs[s] *= v;
}
void launch_scale_prep(const DevProblem& P, const double* d, double* dS, cudaStream_t st) {
    k_scale_prep<<<(P.ldS + 255) / 256, 256, 0, st>>>(P, d, dS);
    count_launch();
}
// camera-side step from the solution in S order: pc[x column] = xs[s] (* d).  The blocks behind the first ldS threads
// fill the dense per-image table pEO[image][6] of the EO step (0 for fixed elements) that the back-substitution
// gathers with three 16-byte loads per observation instead of a column lookup plus a second gather.
__global__ void k_unpermute(DevProblem P, const double* __restrict__ xs, const double* __restrict__ d,
                            double* __restrict__ pc, double* __restrict__ pEO, int nbS) {
    if ((int)blockIdx.x < nbS) {
        const int s = blockIdx.x * blockDim.x + threadIdx.x;
        if (s >= P.ldS) return;
        const int c = P.s2x[s];
        if (c >= 0) pc[c] = d ? xs[s] * d[c] : xs[s];
        return;
    }
    const int t = (blockIdx.x - nbS) * blockDim.x + threadIdx.x;
    if (t >= 6 * P.nImg) return;
    const int si = P.eo_s[t];
    double v = 0.0;
    if (si >= 0) v = d ? xs[si] * d[P.eo_col[t]] : xs[si];
    pEO[t] = v;
}
void launch_unpermute(const DevProblem& P, const double* xs, const double* d, double* pc, double* pEO, cudaStream_t st) {
    const int nbS = (P.ldS + 255) / 256, nbE = pEO ? (6 * P.nImg + 255) / 256 : 0;
    k_unpermute<<<nbS + nbE, 256, 0, st>>>(P, xs, d, pc, pEO, nbS);
    count_launch();
}

// back-substitution for the object points of `list` (those with more than DBAT_PSB observations), one thread per
// point; p[0:nC] must already hold the camera/IO step.
// By-product (stats != nullptr): this block's share of  p'J'Jp = |Jp|^2  and  r'Jp = g'p  over the point
// columns, from the blocks already in registers - with a_j = W~_j' p_c and the UNDAMPED V_j, g_j:
//     |Jp|^2 = p_c' N_cc p_c + sum_j ( p_j' V_j p_j + 2 p_j' a_j ),     r'Jp = g_c' p_c + sum_j g_j' p_j
// (levenberg_marquardt.m:162 forms J*p explicitly; same number, one pass over the observations less).
__global__ void __launch_bounds__(128) k_backsub(DevProblem P, double lambda, double* __restrict__ p,
                                                  double* __restrict__ stats, int statStride,
                                                  const int* __restrict__ list, int nList) {
    __shared__ double red[2][4];
    const int jj = blockIdx.x * blockDim.x + threadIdx.x;
    const int j = jj < nList ? list[jj] : P.nOP;
    double jp2 = 0.0, rjp = 0.0;
    if (j < P.nOP) {
        const int* opc = P.op_col + 3 * (size_t)j;
        if (!(opc[0] < 0 && opc[1] < 0 && opc[2] < 0)) {
            const double* rec = P.pt + (size_t)j * DBAT_PT_STRIDE;
            double Vi[6];
            point_inverse(rec, opc, lambda, Vi);
            double a[3] = {0.0, 0.0, 0.0};                  // W~_j' p_c
#pragma unroll
            for (int s = 0; s < DBAT_NSLOT; ++s) {
                const int c = P.sh_col[s];
                if (c < 0) continue;
                const double pv = p[c];
                const double* ws = rec + DBAT_PT_WSH + 3 * s;
                a[0] += ws[0] * pv; a[1] += ws[1] * pv; a[2] += ws[2] * pv;
            }
            const int o0 = P.pt_start[j], o1 = P.pt_start[j + 1];
            for (int ob = o0; ob < o1; ++ob) {
                const int* ec = P.eo_col + 6 * (size_t)P.img_pm[ob];
                const double* Wo = P.W + (size_t)ob * DBAT_W_STRIDE;
#pragma unroll
                for (int e = 0; e < 6; ++e) {
                    const int c = ec[e];
                    if (c < 0) continue;
                    const double pv = p[c];
                    a[0] += Wo[3 * e] * pv; a[1] += Wo[3 * e + 1] * pv; a[2] += Wo[3 * e + 2] * pv;
                }
            }
            const double t[3] = {-rec[6] - a[0], -rec[7] - a[1], -rec[8] - a[2]};
            double y[3];
            symv3(Vi, t, y);
#pragma unroll
            for (int e = 0; e < 3; ++e) if (opc[e] >= 0) p[opc[e]] = y[e]; else y[e] = 0.0;
            const double Vy0 = rec[0] * y[0] + rec[1] * y[1] + rec[2] * y[2];
            const double Vy1 = rec[1] * y[0] + rec[3] * y[1] + rec[4] * y[2];
            const double Vy2 = rec[2] * y[0] + rec[4] * y[1] + rec[5] * y[2];
            jp2 = y[0] * (Vy0 + 2.0 * a[0]) + y[1] * (Vy1 + 2.0 * a[1]) + y[2] * (Vy2 + 2.0 * a[2]);
            rjp = rec[6] * y[0] + rec[7] * y[1] + rec[8] * y[2];
        }
    }
    if (stats) {                                             // fixed-order block sums: bit-reproducible
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) { jp2 += __shfl_xor_sync(0xffffffffu, jp2, o); rjp += __shfl_xor_sync(0xffffffffu, rjp, o); }
        if ((threadIdx.x & 31) == 0) { red[0][threadIdx.x >> 5] = jp2; red[1][threadIdx.x >> 5] = rjp; }
        __syncthreads();
        if (threadIdx.x == 0) {
            stats[blockIdx.x] = (red[0][0] + red[0][1]) + (red[0][2] + red[0][3]);
            stats[statStride + blockIdx.x] = (red[1][0] + red[1][1]) + (red[1][2] + red[1][3]);
        }
    }
}
// The same back-substitution with one thread per OBSERVATION for all other points: the blocks of
// k_point_side_obs (whole points, at most DBAT_PSB observations).  Phase 1: thread o reads its cross block W_o
// (144 contiguous bytes, consecutive threads consecutive blocks: fully coalesced) and the six EO entries of p_c
// of its image and leaves a_o = W_o' p_c in shared memory.  Phase 2: one thread per point adds the a_o of its
// observations in image order, the shared IO part, solves with (V_j + lambda I)^-1 and forms the |Jp|^2 / r'Jp terms.
// The EO step of the observation's image comes from the dense table pEO (three 16-byte loads instead of a column
// lookup and a dependent gather); the lines phase 2 will need (point record, column map) start towards L1 at once and
// the shared IO step is read once per block.  Measured and dropped: the point's (V + lambda I)^-1 before the barrier
// (more registers, fewer resident blocks: slower).
__global__ void __launch_bounds__(DBAT_PSB) k_backsub_obs(DevProblem P, double lambda, double* __restrict__ p,
                                                           const double* __restrict__ pEO,
                                                           double* __restrict__ stats, int statStride) {
    __shared__ double ao[DBAT_PSB * 3];
    __shared__ double red[2][DBAT_PSB / 32];
    __shared__ double psh[DBAT_NSLOT + 2];
    __shared__ int pshOk[DBAT_NSLOT + 2];
    const int tid = threadIdx.x;
    const int p0 = P.psb_pt[2 * blockIdx.x], p1 = P.psb_pt[2 * blockIdx.x + 1];
    const int ob0 = P.pt_start[p0], nob = P.pt_start[p1] - ob0;
    if (p0 + tid < p1) {
        const char* rec = reinterpret_cast<const char*>(P.pt + (size_t)(p0 + tid) * DBAT_PT_STRIDE);
#pragma unroll
        for (int b = 0; b < DBAT_PT_STRIDE * 8; b += 128) asm volatile("prefetch.global.L1 [%0];" :: "l"(rec + b));
        asm volatile("prefetch.global.L1 [%0];" :: "l"(rec + DBAT_PT_STRIDE * 8 - 8));      // the record's last line when it straddles a fifth one
        asm volatile("prefetch.global.L1 [%0];" :: "l"(P.op_col + 3 * (size_t)(p0 + tid)));
    }
    if (tid >= DBAT_PSB - DBAT_NSLOT) {                          // the shared IO step, once per block
        const int s = tid - (DBAT_PSB - DBAT_NSLOT);
        const int c = P.sh_col[s];
        psh[s] = c >= 0 ? p[c] : 0.0;
        pshOk[s] = c >= 0;
    }
    if (tid < nob) {
        const int ob = ob0 + tid;
        const double2* Wo = reinterpret_cast<const double2*>(P.W + (size_t)ob * DBAT_W_STRIDE);
        double w[18];
#pragma unroll
        for (int q = 0; q < 9; ++q) { const double2 t = Wo[q]; w[2 * q] = t.x; w[2 * q + 1] = t.y; }
        double a0 = 0.0, a1 = 0.0, a2 = 0.0;
        const double2* pe = reinterpret_cast<const double2*>(pEO + 6 * (size_t)P.img_pm[ob]);
        const double2 e01 = pe[0], e23 = pe[1], e45 = pe[2];
        const double pv[6] = {e01.x, e01.y, e23.x, e23.y, e45.x, e45.y};
#pragma unroll
        for (int e = 0; e < 6; ++e) { a0 += w[3 * e] * pv[e]; a1 += w[3 * e + 1] * pv[e]; a2 += w[3 * e + 2] * pv[e]; }
        ao[3 * tid] = a0; ao[3 * tid + 1] = a1; ao[3 * tid + 2] = a2;
    }
    __syncthreads();
    double jp2 = 0.0, rjp = 0.0;
    const int j = p0 + tid;
    if (j < p1) {
        const int* opc = P.op_col + 3 * (size_t)j;
        if (!(opc[0] < 0 && opc[1] < 0 && opc[2] < 0)) {
            const double* rec = P.pt + (size_t)j * DBAT_PT_STRIDE;
            double Vi[6];
            point_inverse(rec, opc, lambda, Vi);
            double a[3] = {0.0, 0.0, 0.0};
#pragma unroll
            for (int s = 0; s < DBAT_NSLOT; ++s) {
                if (!pshOk[s]) continue;
                const double pv = psh[s];
                const double* ws = rec + DBAT_PT_WSH + 3 * s;
                a[0] += ws[0] * pv; a[1] += ws[1] * pv; a[2] += ws[2] * pv;
            }
            for (int r = P.pt_start[j] - ob0; r < P.pt_start[j + 1] - ob0; ++r) { a[0] += ao[3 * r]; a[1] += ao[3 * r + 1]; a[2] += ao[3 * r + 2]; }
            const double t[3] = {-rec[6] - a[0], -rec[7] - a[1], -rec[8] - a[2]};
            double y[3];
            symv3(Vi, t, y);
#pragma unroll
            for (int e = 0; e < 3; ++e) if (opc[e] >= 0) p[opc[e]] = y[e]; else y[e] = 0.0;
            const double Vy0 = rec[0] * y[0] + rec[1] * y[1] + rec[2] * y[2];
            const double Vy1 = rec[1] * y[0] + rec[3] * y[1] + rec[4] * y[2];
            const double Vy2 = rec[2] * y[0] + rec[4] * y[1] + rec[5] * y[2];
            jp2 = y[0] * (Vy0 + 2.0 * a[0]) + y[1] * (Vy1 + 2.0 * a[1]) + y[2] * (Vy2 + 2.0 * a[2]);
            rjp = rec[6] * y[0] + rec[7] * y[1] + rec[8] * y[2];
        }
    }
    if (stats) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) { jp2 += __shfl_xor_sync(0xffffffffu, jp2, o); rjp += __shfl_xor_sync(0xffffffffu, rjp, o); }
        if ((tid & 31) == 0) { red[0][tid >> 5] = jp2; red[1][tid >> 5] = rjp; }
        __syncthreads();
        if (tid == 0) {
            double s0 = 0.0, s1 = 0.0;
#pragma unroll
            for (int w = 0; w < DBAT_PSB / 32; ++w) { s0 += red[0][w]; s1 += red[1][w]; }
            stats[blockIdx.x] = s0; stats[statStride + blockIdx.x] = s1;
        }
    }
}
// camera part of p'J'Jp and g'p: per image (p_io; p_eo_i)' G_i (p_io; p_eo_i) from the per-image Grams (their IO x IO
// blocks add up to the shared block), the prior terms of the camera-side columns by image 0's thread block
__global__ void __launch_bounds__(128) k_jp_cam(DevProblem P, const double* __restrict__ p,
                                                 const double* __restrict__ camDiag, const double* __restrict__ camG,
                                                 double* __restrict__ stats) {
    __shared__ double red[2][4];
    __shared__ double vs[4][DBAT_NSLOT + 6 + 2];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int i = blockIdx.x * 4 + warp;                      // one warp per image
    constexpr int NV = DBAT_NSLOT + 6;
    double jp2 = 0.0, rjp = 0.0;
    if (i < P.nImg) {
        if (lane < NV) {
            const int c = P.cam_colx[(size_t)DBAT_NCAM * i + lane];
            vs[warp][lane] = c >= 0 ? p[c] : 0.0;
        }
        __syncwarp();
        const double* G = P.imgG + (size_t)i * DBAT_GSZ;
        for (int e = lane; e < NV * NV; e += 32) {
            const int a = e / NV, b = e - a * NV;
            jp2 += vs[warp][a] * gram_at(G, a, b) * vs[warp][b];
        }
        if (lane < NV) rjp += vs[warp][lane] * gram_at(G, lane, DBAT_COL_R);
    }
    for (int c = blockIdx.x * blockDim.x + threadIdx.x; c < P.nC; c += gridDim.x * blockDim.x) {   // prior rows
        jp2 += camDiag[c] * p[c] * p[c];
        rjp += camG[c] * p[c];
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { jp2 += __shfl_xor_sync(0xffffffffu, jp2, o); rjp += __shfl_xor_sync(0xffffffffu, rjp, o); }
    if (lane == 0) { red[0][warp] = jp2; red[1][warp] = rjp; }
    __syncthreads();
    if (threadIdx.x == 0) {
        stats[blockIdx.x] = (red[0][0] + red[0][1]) + (red[0][2] + red[0][3]);
        stats[gridDim.x + blockIdx.x] = (red[1][0] + red[1][1]) + (red[1][2] + red[1][3]);
    }
}
// sums of two partial arrays (a[0..n), a[n..2n)) into out[0], out[1]; one block per array pair, fixed order, four
// independent chains per thread (the loop is latency-bound).  Block 1 (if launched) does the same for (b, nb) -> out[2..3].
__global__ void __launch_bounds__(1024) k_sum_pair(const double* __restrict__ a, int n, double* __restrict__ out,
                                                    const double* __restrict__ b, int nb) {
    __shared__ double sm[2][32];
    if (blockIdx.x == 1) { a = b; n = nb; out += 2; }
    double s0 = 0.0, s1 = 0.0, t0 = 0.0, t1 = 0.0, u0 = 0.0, u1 = 0.0, v0 = 0.0, v1 = 0.0;
    int k = threadIdx.x;
    for (; k + 3072 < n; k += 4096) {
        s0 += a[k]; s1 += a[n + k]; t0 += a[k + 1024]; t1 += a[n + k + 1024];
        u0 += a[k + 2048]; u1 += a[n + k + 2048]; v0 += a[k + 3072]; v1 += a[n + k + 3072];
    }
    for (; k < n; k += 1024) { s0 += a[k]; s1 += a[n + k]; }
    s0 = (s0 + t0) + (u0 + v0); s1 = (s1 + t1) + (u1 + v1);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { s0 += __shfl_xor_sync(0xffffffffu, s0, o); s1 += __shfl_xor_sync(0xffffffffu, s1, o); }
    if ((threadIdx.x & 31) == 0) { sm[0][threadIdx.x >> 5] = s0; sm[1][threadIdx.x >> 5] = s1; }
    __syncthreads();
    if (threadIdx.x < 32) {
        s0 = sm[0][threadIdx.x]; s1 = sm[1][threadIdx.x];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) { s0 += __shfl_xor_sync(0xffffffffu, s0, o); s1 += __shfl_xor_sync(0xffffffffu, s1, o); }
        if (threadIdx.x == 0) { out[0] = s0; out[1] = s1; }
    }
}
// p = [pc ; back-substituted points].  jpOut (4 doubles, may be null): [0..1] point part of |Jp|^2, r'Jp (a multi-rank
// run sums these over the ranks), [2..3] the camera part (identical on every rank).
void launch_backsub(const DevProblem& P, double lambda, const double* pc, const double* pEO, double* p, double* partial,
                    const double* camDiag, const double* camG, double* jpOut, cudaStream_t st,
                    cudaStream_t st2, cudaEvent_t evFork, cudaEvent_t evJoin) {
    if (pc != p) cudaMemcpyAsync(p, pc, sizeof(double) * P.nC, cudaMemcpyDeviceToDevice, st);
    // number of per-block partial pairs the point kernels will write (the camera part's partials follow them)
    int nb = 0;
    const int nbBig = P.nPsbig > 0 ? (P.nPsbig + 127) / 128 : 0;
    const bool general = P.nOP > 0 && P.ioGeneral;
    if (general) nb = (P.nOP + 127) / 128;        // launch_backsub_gen: one warp-free block per 128 points
    else if (P.nOP > 0) nb = P.nPsb + nbBig;
    const int nbc = (P.nImg + 3) / 4;
    const bool side = jpOut && st2 && evFork && evJoin;
    if (side) {
        // the camera part of |Jp|^2, r'Jp needs only p_c and the Grams: it runs beside the back-substitution
        cudaEventRecord(evFork, st);
        cudaStreamWaitEvent(st2, evFork, 0);
        k_jp_cam<<<nbc, 128, 0, st2>>>(P, p, camDiag, camG, partial + 2 * nb);
        cudaEventRecord(evJoin, st2);
        count_launch();
    }
    if (general) {
        launch_backsub_gen(P, lambda, p, jpOut ? partial : nullptr, st);
    } else if (P.nOP > 0) {
        if (P.nPsb > 0) { k_backsub_obs<<<P.nPsb, DBAT_PSB, 0, st>>>(P, lambda, p, pEO, jpOut ? partial : nullptr, nb); count_launch(); }
        if (nbBig > 0) { k_backsub<<<nbBig, 128, 0, st>>>(P, lambda, p, jpOut ? partial + P.nPsb : nullptr, nb, P.psbig, P.nPsbig); count_launch(); }
    }
    if (jpOut) {
        if (side) cudaStreamWaitEvent(st, evJoin, 0);
        else { k_jp_cam<<<nbc, 128, 0, st>>>(P, p, camDiag, camG, partial + 2 * nb); count_launch(); }
        if (nb == 0) cudaMemsetAsync(jpOut, 0, 2 * sizeof(double), st);
        // block 0: point part -> jpOut[0..1]; block 1: camera part -> jpOut[2..3]
        if (nb > 0) k_sum_pair<<<2, 1024, 0, st>>>(partial, nb, jpOut, partial + 2 * nb, nbc);
        else k_sum_pair<<<1, 1024, 0, st>>>(partial + 2 * nb, nbc, jpOut + 2, nullptr, 0);
        count_launch();
    }
}

// ---------------------------------------------------------------------------------------------
// deterministic vector helpers
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ double warp_sum2(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__global__ void k_dot_partial(const double* __restrict__ a, const double* __restrict__ b, int n,
                              double* __restrict__ partial) {
    __shared__ double sm[32];
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    double v = (k < n) ? a[k] * (b ? b[k] : 1.0) : 0.0;
    v = warp_sum2(v);
    if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x < 32) {
        double t = threadIdx.x < (blockDim.x >> 5) ? sm[threadIdx.x] : 0.0;
        t = warp_sum2(t);
        if (threadIdx.x == 0) partial[blockIdx.x] = t;
    }
}
__global__ void k_final_sum2(const double* __restrict__ partial, int n, double* __restrict__ out, int slot) {
    __shared__ double sm[32];
    double s = 0.0;
    for (int k = threadIdx.x; k < n; k += blockDim.x) s += partial[k];
    s = warp_sum2(s);
    if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x < 32) {
        double t = threadIdx.x < (blockDim.x >> 5) ? sm[threadIdx.x] : 0.0;
        t = warp_sum2(t);
        if (threadIdx.x == 0) out[slot] = t;
    }
}
void launch_dot(const double* a, const double* b, int n, double* partial, double* scal, int slot,
                cudaStream_t st) {
    const int nb = (n + 255) / 256;
    if (nb > 0) k_dot_partial<<<nb, 256, 0, st>>>(a, b, n, partial);
    k_final_sum2<<<1, 256, 0, st>>>(partial, nb, scal, slot);
    count_launch(2);
}
void launch_vec_ops_sum(const double* a, int n, double* partial, double* scal, int slot, cudaStream_t st) {
    launch_dot(a, nullptr, n, partial, scal, slot, st);
}
__global__ void k_axpy(double alpha, const double* __restrict__ x, const double* __restrict__ y,
                       double* __restrict__ out, int n) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k < n) out[k] = y[k] + alpha * x[k];
}
void launch_axpy(double alpha, const double* x, const double* y, double* out, int n, cudaStream_t st) {
    if (n <= 0) return;
    k_axpy<<<(n + 255) / 256, 256, 0, st>>>(alpha, x, y, out, n);
    count_launch();
}
__global__ void k_inv_sqrt(const double* __restrict__ in, double* __restrict__ out, int n) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k < n) out[k] = 1.0 / sqrt(in[k]);
}
void launch_inv_sqrt(const double* in, double* out, int n, cudaStream_t st) {
    if (n <= 0) return;
    k_inv_sqrt<<<(n + 255) / 256, 256, 0, st>>>(in, out, n);
    count_launch();
}
__global__ void k_mul(const double* __restrict__ a, const double* __restrict__ b, double* __restrict__ out, int n) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k < n) out[k] = a[k] * b[k];
}
void launch_mul(const double* a, const double* b, double* out, int n, cudaStream_t st) {
    if (n <= 0) return;
    k_mul<<<(n + 255) / 256, 256, 0, st>>>(a, b, out, n);
    count_launch();
}
