// schur_wide.cu — Schur reduction of the wide points (estimated points with more than DBAT_GRP_MAXM rays, which the
// window kernels of schur_win.cu do not group), without atomics.
//
// Same formulation as the window path: with M_j = inv(chol(V_j + lambda I)) (unit diagonal for fixed coordinates),
// Z_o = M_j W_o' (3 x 6) for every observation o of point j, zsh_j = M_j Wsh_j' and zg_j = M_j g_j,
//   S(A,B)   -= sum_j Z_jA' Z_jB        S(sh,A) -= sum_j zsh_j' Z_jA        S(sh,sh) -= sum_j zsh_j' zsh_j
//   rhs(A)   += sum_j Z_jA' zg_j        rhs(sh) += sum_j zsh_j' zg_j
// in two kernels:
//
//   k_wide_stage   Z_o of every wide observation (one thread each) and, one CTA per DBAT_WIDE_SSPART wide points,
//                  [zsh_j zg_j] and the partial shared x shared table of those points.
//   k_wide_reduce  one warp per camera-pair block that wide points touch: walks the shorter of the two images' lists
//                  (wide observations in ascending point order), finds each point in the other list by binary search
//                  and adds Z_jA' Z_jB of the common points in ascending point order on the FP64 tensor pipe (DMMA
//                  m8n8k4, K = the 3 coordinates of one point).  One warp per image for its shared-IO x EO rows and
//                  rhs(A), over its list in the same order.  One CTA adds the partial tables in order into
//                  wide_shAcc, which k_schur_ss_apply adds to the shared x shared block.
//
// Every entry of S and of the rhs gets its wide-point terms in an order fixed by the plan, from one thread, so the
// result is bit-reproducible.  The index is linear in the wide observations plus one entry per touched pair block.
#include "kernels.cuh"
#include "launch.h"

#define WIDE_WARPS 8                     // warps per CTA of k_wide_reduce
static_assert(DBAT_WIDE_SSPART == 16, "k_wide_stage: one CTA of 256 threads = 16 points x 16 shared rows");

__device__ __forceinline__ void dmma_wide(double& c0, double& c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}

// inv(chol(V_j + lambda I)) = [m00; m10 m11; m20 m21 m22], the arithmetic of k_point_minv (schur_win.cu)
__device__ __forceinline__ void wide_minv(const double* __restrict__ rec, const int* __restrict__ opc, double lambda,
                                          double m[6]) {
    double a00 = rec[0], a01 = rec[1], a02 = rec[2], a11 = rec[3], a12 = rec[4], a22 = rec[5];
    a00 = opc[0] >= 0 ? a00 + lambda : 1.0;
    a11 = opc[1] >= 0 ? a11 + lambda : 1.0;
    a22 = opc[2] >= 0 ? a22 + lambda : 1.0;
    const double l00 = sqrt(a00);
    const double l10 = a01 / l00, l20 = a02 / l00;
    const double l11 = sqrt(a11 - l10 * l10);
    const double l21 = (a12 - l20 * l10) / l11;
    const double l22 = sqrt(a22 - l20 * l20 - l21 * l21);
    const double m00 = 1.0 / l00, m11 = 1.0 / l11, m22 = 1.0 / l22;
    m[0] = m00; m[1] = -l10 * m00 * m11; m[2] = m11;
    m[4] = -l21 * m11 * m22;
    m[3] = -(l20 * m00 + l21 * m[1]) * m22;
    m[5] = m22;
}

// z = M w for one row w of a cross block (the products of cell_put in schur_win.cu)
__device__ __forceinline__ void wide_mw(const double m[6], double w0, double w1, double w2, double z[3]) {
    z[0] = w0 * m[0];
    z[1] = w0 * m[1] + w1 * m[2];
    z[2] = w0 * m[3] + w1 * m[4] + w2 * m[5];
}

// blocks [0, nbZ): Z_o of wide observation blockIdx.x * 256 + t; blocks [nbZ, ...): part q of the wide points
__global__ void __launch_bounds__(256) k_wide_stage(DevProblem P, double lambda, int nbZ) {
    const int t = threadIdx.x;
    if ((int)blockIdx.x < nbZ) {
        const int w = blockIdx.x * 256 + t;
        if (w >= P.nWObs) return;
        const int o = P.wide_o[w], j = P.pt_pm[o];
        double m[6];
        wide_minv(P.pt + (size_t)j * DBAT_PT_STRIDE, P.op_col + 3 * (size_t)j, lambda, m);
        const double2* Wo = reinterpret_cast<const double2*>(P.W + (size_t)o * DBAT_W_STRIDE);
        double wv[18];
#pragma unroll
        for (int k = 0; k < 9; ++k) { const double2 v = Wo[k]; wv[2 * k] = v.x; wv[2 * k + 1] = v.y; }
        double zo[18];                                     // [k][a]
#pragma unroll
        for (int a = 0; a < 6; ++a) {
            double z[3];
            wide_mw(m, wv[3 * a], wv[3 * a + 1], wv[3 * a + 2], z);
            zo[a] = z[0]; zo[6 + a] = z[1]; zo[12 + a] = z[2];
        }
        double2* out = reinterpret_cast<double2*>(P.wide_Z + (size_t)w * 18);
#pragma unroll
        for (int k = 0; k < 9; ++k) out[k] = make_double2(zo[2 * k], zo[2 * k + 1]);
        return;
    }
    __shared__ double zs[DBAT_WIDE_SSPART][3][16];
    const int q = blockIdx.x - nbZ;
    const int pt = t >> 4, s = t & 15;                      // 16 points x 16 rows (14 IO slots, gradient, zero)
    const int jb = q * DBAT_WIDE_SSPART + pt;
    double z[3] = {0.0, 0.0, 0.0};
    if (jb < P.nBig) {
        const int j = P.big_pt[jb];
        const double* rec = P.pt + (size_t)j * DBAT_PT_STRIDE;
        double m[6];
        wide_minv(rec, P.op_col + 3 * (size_t)j, lambda, m);
        if (s < DBAT_NSLOT) wide_mw(m, rec[DBAT_PT_WSH + 3 * s], rec[DBAT_PT_WSH + 3 * s + 1], rec[DBAT_PT_WSH + 3 * s + 2], z);
        else if (s == DBAT_NSLOT) wide_mw(m, rec[6], rec[7], rec[8], z);
        double* out = P.wide_Zsh + (size_t)jb * 48;
        out[s] = z[0]; out[16 + s] = z[1]; out[32 + s] = z[2];
    }
    zs[pt][0][s] = z[0]; zs[pt][1][s] = z[1]; zs[pt][2][s] = z[2];
    __syncthreads();
    const int a = t >> 4, b = t & 15;
    double acc = 0.0;
#pragma unroll
    for (int p = 0; p < DBAT_WIDE_SSPART; ++p) acc += zs[p][0][a] * zs[p][0][b] + zs[p][1][a] * zs[p][1][b] + zs[p][2][a] * zs[p][2][b];
    P.wide_ssPart[(size_t)q * 256 + t] = acc;
}

// blocks [0, nbP): one warp per pair block; [nbP, nbP + nbI): one warp per image; the last block: the shared table
__global__ void __launch_bounds__(32 * WIDE_WARPS) k_wide_reduce(DevProblem P, int nbP, int nbI, int nPart) {
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const int fr = lane >> 2, fk = lane & 3;               // DMMA fragment row / k
    const bool on = fr < 6 && fk < 3;                      // lanes holding a coordinate x EO element of Z
    const int zoff = fk * 6 + fr;
    const double* __restrict__ Z = P.wide_Z;
    if ((int)blockIdx.x < nbP) {
        const int pr = blockIdx.x * WIDE_WARPS + warp;
        if (pr >= P.nWPair) return;
        const int iA = P.wpair[2 * pr], iB = P.wpair[2 * pr + 1];
        const int a0 = P.wimg_ptr[iA], a1 = P.wimg_ptr[iA + 1];
        double c0 = 0.0, c1 = 0.0;                         // C[fr][2 fk], C[fr][2 fk + 1] of the 6 x 6 block
        if (iA == iB) {
            for (int q = a0; q < a1; ++q) {
                const double z = on ? Z[(size_t)P.wimg_w[q] * 18 + zoff] : 0.0;
                dmma_wide(c0, c1, z, z);
            }
        } else {
            const int b0 = P.wimg_ptr[iB], b1 = P.wimg_ptr[iB + 1];
            const bool aShort = a1 - a0 <= b1 - b0;
            const int s0 = aShort ? a0 : b0, s1 = aShort ? a1 : b1, l1 = aShort ? b1 : a1;
            int lo = aShort ? b0 : a0;
            for (int base = s0; base < s1; base += 32) {
                // lane: one point of the short list, its position in the long one (both lists ascend in point)
                const int q = base + lane;
                int ws = -1, wl = -1, pos = l1;
                if (q < s1) {
                    const int pt = P.wimg_pt[q];
                    int l = lo, h = l1;
                    while (l < h) { const int mid = (l + h) >> 1; if (P.wimg_pt[mid] < pt) l = mid + 1; else h = mid; }
                    pos = l;
                    if (l < l1 && P.wimg_pt[l] == pt) { ws = P.wimg_w[q]; wl = P.wimg_w[l]; }
                }
                lo = __shfl_sync(0xffffffffu, pos, 31);
                // the common points of this chunk in ascending lane (= point) order; the next one's loads are issued
                // before the current product
                unsigned mk = __ballot_sync(0xffffffffu, ws >= 0);
                if (!mk) continue;
                auto load = [&](int src, double& za, double& zb) {
                    const int xs = __shfl_sync(0xffffffffu, ws, src), xl = __shfl_sync(0xffffffffu, wl, src);
                    const int wa = aShort ? xs : xl, wb = aShort ? xl : xs;
                    za = on ? Z[(size_t)wa * 18 + zoff] : 0.0;
                    zb = on ? Z[(size_t)wb * 18 + zoff] : 0.0;
                };
                double za, zb;
                load(__ffs(mk) - 1, za, zb);
                mk &= mk - 1;
                while (mk) {
                    double na, nb;
                    load(__ffs(mk) - 1, na, nb);
                    mk &= mk - 1;
                    dmma_wide(c0, c1, za, zb);
                    za = na; zb = nb;
                }
                dmma_wide(c0, c1, za, zb);
            }
        }
        if (on) {
            const int row = P.eo_s[6 * (size_t)iA + fr];
            if (row < 0) return;
            const int col0 = P.eo_s[6 * (size_t)iB + 2 * fk], col1 = P.eo_s[6 * (size_t)iB + 2 * fk + 1];
            if (col0 >= 0 && (iA != iB || col0 <= row)) *tc_at(P.T, row, col0) -= c0;
            if (col1 >= 0 && (iA != iB || col1 <= row)) *tc_at(P.T, row, col1) -= c1;
        }
        return;
    }
    if ((int)blockIdx.x < nbP + nbI) {
        // rows s = 0..15 (two 8-row tiles) x EO element a: sum over the image's wide observations of zsh_j' Z_o
        const int img = (blockIdx.x - nbP) * WIDE_WARPS + warp;
        if (img >= P.nImg) return;
        double c00 = 0.0, c01 = 0.0, c10 = 0.0, c11 = 0.0;
        for (int q = P.wimg_ptr[img]; q < P.wimg_ptr[img + 1]; ++q) {
            const double* zsh = P.wide_Zsh + (size_t)P.wimg_pt[q] * 48 + fk * 16 + fr;
            const double zb = on ? Z[(size_t)P.wimg_w[q] * 18 + zoff] : 0.0;
            const double za0 = fk < 3 ? zsh[0] : 0.0, za1 = fk < 3 ? zsh[8] : 0.0;
            dmma_wide(c00, c01, za0, zb);
            dmma_wide(c10, c11, za1, zb);
        }
        if (fk >= 3) return;
        const double v[2][2] = {{c00, c01}, {c10, c11}};
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            const int col = P.eo_s[6 * (size_t)img + 2 * fk + e];
            if (col < 0) continue;
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int s = 8 * h + fr;
                if (s < DBAT_NSLOT) {
                    const int srow = P.sh_s[s];
                    if (srow >= 0) *tc_at(P.T, srow, col) -= v[h][e];
                } else if (s == DBAT_NSLOT) {
                    P.rhs[col] += v[h][e];
                }
            }
        }
        return;
    }
    // shared x shared table and rhs(sh) in k_schur_ss_apply's layout [a][b], b = NSLOT: the gradient column
    if (t < DBAT_NSLOT * (DBAT_NSLOT + 1)) {
        const int a = t / (DBAT_NSLOT + 1), b = t - a * (DBAT_NSLOT + 1);
        double s = 0.0;
        for (int k = 0; k < nPart; ++k) s += P.wide_ssPart[(size_t)k * 256 + a * 16 + b];
        P.wide_shAcc[t] = s;
    }
}

void launch_schur_wide(const DevProblem& P, double lambda, cudaStream_t st) {
    if (P.nBig <= 0) return;
    const int nbZ = (P.nWObs + 255) / 256;
    const int nPart = (P.nBig + DBAT_WIDE_SSPART - 1) / DBAT_WIDE_SSPART;
    k_wide_stage<<<nbZ + nPart, 256, 0, st>>>(P, lambda, nbZ);
    const int nbP = (P.nWPair + WIDE_WARPS - 1) / WIDE_WARPS, nbI = (P.nImg + WIDE_WARPS - 1) / WIDE_WARPS;
    k_wide_reduce<<<nbP + nbI + 1, 32 * WIDE_WARPS, 0, st>>>(P, nbP, nbI, nPart);
    count_launch(2);
}
