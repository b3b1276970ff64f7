// schur_win.cu — Schur reduction onto the camera system without atomics (default path).
//
//   S -= sum_j W~_j (V_j + lambda I)^-1 W~_j',   rhs += sum_j W~_j (V_j + lambda I)^-1 g_j
// (the point elimination behind `(JTJ+lambda*I)\(-JTr)`, code/bundle/lsa/levenberg_marquardt.m:119, in the block
// form of SURVEY.md Appendix A).  The north star asks for a deterministic segmented reduction keyed by an index
// built once; this is it, in two kernels:
//
//   k_schur_win     one CTA per CLUSTER of object points.  Points are sorted by their image lists (create), cut into
//                   groups of <= 14 neighbours whose lists have a union of <= 12 images, and runs of groups whose
//                   unions span <= 20 images (the window) form a cluster.  Per group: with (V + lambda I)^-1 = M'M
//                   (M = inverse Cholesky factor, k_point_minv) the update is the symmetric product Z Z' of
//                   Z = [W~ ; Wsh ; g'] M' - ONE operand in shared memory, staged with the zeros of the images a
//                   point does not see written explicitly (no clearing pass), contracted on the FP64 tensor pipe
//                   (DMMA m8n8k4; one A fragment feeds up to three tiles).  The tiles are added to the cluster's
//                   window accumulator in shared memory (lower-triangular 6 x 6 blocks by window slot; every entry
//                   has one owner lane per group, groups are separated by CTA barriers: fixed order).  At the end
//                   the CTA copies its window image to a staging buffer - coalesced, no atomics.
//   k_schur_reduce  one thread per entry of every camera-pair block of S: adds the images of the clusters that
//                   hold the block in the order of a CSR index built at create, and subtracts the sum from the
//                   tile of S.  Same for the shared-IO x EO rows (per image) and the shared x shared table.
//
// S is touched once per entry, and the result is bit-reproducible.  Points with more than DBAT_GRP_MAXM rays are not
// grouped: schur_wide.cu adds them, also in a fixed order, before these kernels run.
#include <algorithm>
#include <cstdio>
#include <vector>
#include "kernels.cuh"
#include "launch.h"

#ifndef WIN_TH
#define WIN_TH 256
#endif
#ifndef WIN_UNIT
#define WIN_UNIT 3                       // column tiles per work unit (they share the A fragment)
#endif
#define WIN_SHLD (6 * WIN_MAXW)          // row stride of the shared-row accumulator
#define WIN_NBLK (WIN_MAXW * (WIN_MAXW + 1) / 2)
#define WIN_ACC (WIN_NBLK * 36)
#define WIN_MAXRT ((6 * WIN_MAXW + 7) / 8)         // 15 row tiles of camera rows at most
#define WIN_MAXUNIT 96
#define WIN_SSPART 256                   // clusters per partial sum of the shared x shared table

// work units of the tile product for every number RT of camera row tiles: (row tile, first column tile, count <= 3)
// over the lower triangle of the RT camera tiles followed by the two tiles of shared rows (virtual tile indices)
__constant__ unsigned int c_winUnits[WIN_MAXRT + 1][WIN_MAXUNIT];
__constant__ int c_winNUnits[WIN_MAXRT + 1];

static void build_units(unsigned int (*tab)[WIN_MAXUNIT], int* cnt) {
    for (int RT = 0; RT <= WIN_MAXRT; ++RT) {
        std::vector<unsigned int> u;
        for (int ti = 0; ti < RT + 2; ++ti)
            for (int tj = 0; tj <= ti; tj += WIN_UNIT) u.push_back((unsigned)ti | ((unsigned)tj << 8) | ((unsigned)std::min(WIN_UNIT, ti + 1 - tj) << 16));
        std::stable_sort(u.begin(), u.end(), [](unsigned a, unsigned b) { return (a >> 16) > (b >> 16); });   // big units first
        cnt[RT] = (int)u.size();
        for (size_t k = 0; k < u.size(); ++k) tab[RT][k] = u[k];
    }
}

__device__ __forceinline__ void dmma_w(double& c0, double& c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}

// M = inv(chol(V_j + lambda I)) of every grouped point, stored in grp_pt order (a group's factors are contiguous).
// Fixed coordinates carry a unit diagonal and no coupling (their rows of every cross block are zero).
__global__ void k_point_minv(DevProblem P, double lambda) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= P.nCand) return;
    const int j = P.grp_pt[i];
    const double* rec = P.pt + (size_t)j * DBAT_PT_STRIDE;
    const int* opc = P.op_col + 3 * (size_t)j;
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
    const double m10 = -l10 * m00 * m11;
    const double m21 = -l21 * m11 * m22;
    const double m20 = -(l20 * m00 + l21 * m10) * m22;
    double2* o = reinterpret_cast<double2*>(P.winM + 6 * (size_t)i);
    o[0] = make_double2(m00, m10); o[1] = make_double2(m11, m20); o[2] = make_double2(m21, m22);
}

struct WinPrefetch { int4 h; double2 m; };

// row stride of the k-major operand Zt[k][row]: smallest value >= rows with stride = 4 mod 8 (conflict-free
// fragment loads: lanes (fr, fk) of a half warp read Zt[(k0 + fk) * LDR + row0 + fr], fk * LDR mod 16 = 0, 4, 8, 12 in some order)
__host__ __device__ constexpr int win_ldr(int rowsZ) { return ((rowsZ - 4 + 7) / 8) * 8 + 4; }

// one work unit: CNT column tiles against one row tile; k offsets are immediates (LDR is a template parameter)
template <int LDR, int CNT>
__device__ __forceinline__ void win_unit_mma(const double* __restrict__ pa, const double* __restrict__ pb0,
                                             const double* __restrict__ pb1, const double* __restrict__ pb2, int Kp,
                                             double (&c)[3][2]) {
    // even and odd k-steps into separate accumulators: two dependent DMMA chains per tile instead of one
    double d[3][2] = {{0.0, 0.0}, {0.0, 0.0}, {0.0, 0.0}};
#pragma unroll
    for (int ks = 0; ks < (3 * WIN_GP + 3) / 4; ks += 2) {
        if (4 * ks >= Kp) break;
        const double a = pa[4 * ks * LDR];
        dmma_w(c[0][0], c[0][1], a, pb0[4 * ks * LDR]);
        if (CNT > 1) dmma_w(c[1][0], c[1][1], a, pb1[4 * ks * LDR]);
        if (CNT > 2) dmma_w(c[2][0], c[2][1], a, pb2[4 * ks * LDR]);
        if (4 * (ks + 1) < Kp && ks + 1 < (3 * WIN_GP + 3) / 4) {
            const double a2 = pa[4 * (ks + 1) * LDR];
            dmma_w(d[0][0], d[0][1], a2, pb0[4 * (ks + 1) * LDR]);
            if (CNT > 1) dmma_w(d[1][0], d[1][1], a2, pb1[4 * (ks + 1) * LDR]);
            if (CNT > 2) dmma_w(d[2][0], d[2][1], a2, pb2[4 * (ks + 1) * LDR]);
        }
    }
#pragma unroll
    for (int n = 0; n < CNT; ++n) { c[n][0] += d[n][0]; c[n][1] += d[n][1]; }
}

// dynamic shared memory: Zt[3 * WIN_GP + 2][LDR] | Acc[WIN_ACC] | AccSh[16][WIN_SHLD] | AccSS[16][16]
template <int LDR>
__global__ void __launch_bounds__(WIN_TH, 2) k_schur_win(DevProblem P) {
    extern __shared__ __align__(16) double dsm[];
    __shared__ __align__(16) WinHdr s_hdr[3];
    __shared__ __align__(16) double s_M[2][WIN_GP * 6];
    __shared__ int s_rowTab[8 * WIN_MAXRT], s_colTab[4 * WIN_MAXRT], s_colSh[4 * WIN_MAXRT];
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const int fr = lane >> 2, fk = lane & 3;
    const int RTmaxP = (6 * P.grpMaxRays + 7) >> 3;          // camera row tiles of the largest union of the problem
    const int shRow0 = 8 * RTmaxP;                           // the 16 shared rows (14 IO slots, gradient, pad) follow
    constexpr int ZT = (3 * WIN_GP + 2) * LDR;
    double* Zt = dsm;
    double* Acc = Zt + ZT;
    double* AccSh = Acc + WIN_ACC;
    double* AccSS = AccSh + 16 * WIN_SHLD;
    const int clu = P.clu_order[blockIdx.x];                 // largest clusters first
    const int g0 = P.clu_grp[clu], g1 = P.clu_grp[clu + 1];
    const int mw = P.clu_img_off[clu + 1] - P.clu_img_off[clu];
    for (int i = t; i < (ZT + WIN_ACC + 16 * WIN_SHLD + 256) / 2; i += WIN_TH)
        reinterpret_cast<double2*>(dsm)[i] = make_double2(0.0, 0.0);
    // ---- raw cells of a group: cell idx = (point gi, q): q < m - the 6 x 3 cross block of the point in union image
    //      q (zeros if the point does not see it); q = m, m+1, m+2 - shared IO rows 0-5, 6-11, 12-13 + gradient + zero
    //      row.  One cell = 18 doubles = nine 16-byte loads; a group has at most 14 * 15 = 210 cells when its union
    //      holds <= 12 images: one per thread, kept in registers while the previous group's products run.
    auto cell_load = [&](const WinHdr& H, int idx, int mq, unsigned inv, double2 (&w)[9]) {
        const int gi = (int)(((unsigned)idx * inv) >> 24), q = idx - gi * mq;
#pragma unroll
        for (int k = 0; k < 9; ++k) w[k] = make_double2(0.0, 0.0);
        if (q < mq - 3) {
            const int o = H.obsOf[gi][q];
            if (o != 255) {
                const double2* p = reinterpret_cast<const double2*>(P.W + (size_t)(H.ob[gi] + o) * DBAT_W_STRIDE);
#pragma unroll
                for (int k = 0; k < 9; ++k) w[k] = p[k];
            }
        } else {
            const int b = q - (mq - 3);
            const double2* rec = reinterpret_cast<const double2*>(P.pt + (size_t)H.j[gi] * DBAT_PT_STRIDE);
            if (b < 2) {
#pragma unroll
                for (int k = 0; k < 9; ++k) w[k] = rec[5 + 9 * b + k];       // Wsh rows 6b .. 6b+5 (record offset 10 + 18 b)
            } else {
                w[0] = rec[23]; w[1] = rec[24]; w[2] = rec[25];              // Wsh rows 12, 13
                const double2 g01 = rec[3], g2 = rec[4];                     // gradient (record offset 6)
                w[3] = g01; w[4] = make_double2(g2.x, 0.0);
            }
        }
    };
    auto cell_put = [&](const WinHdr& H, const double* Ms, int idx, int mq, unsigned inv, const double2 (&w)[9]) {
        const int gi = (int)(((unsigned)idx * inv) >> 24), q = idx - gi * mq;
        const int row0 = q < mq - 3 ? 6 * q : shRow0 + 6 * (q - (mq - 3));
        const double* Mg = Ms + 6 * gi;                      // m00 m10 m11 m20 m21 m22
        const double m00 = Mg[0], m10 = Mg[1], m11 = Mg[2], m20 = Mg[3], m21 = Mg[4], m22 = Mg[5];
        double* z = Zt + (3 * gi) * LDR + row0;
        const double* wd = reinterpret_cast<const double*>(w);
#pragma unroll
        for (int a = 0; a < 6; ++a) {
            const double w0 = wd[3 * a], w1 = wd[3 * a + 1], w2 = wd[3 * a + 2];
            z[a] = w0 * m00;
            z[LDR + a] = w0 * m10 + w1 * m11;
            z[2 * LDR + a] = w0 * m20 + w1 * m21 + w2 * m22;
        }
    };
    double2 cw[9];
    auto load_cells = [&](const WinHdr& H) {
        const int mq = H.m + 3;
        const unsigned inv = (0x1000000u + mq - 1) / mq;
        if (t < H.ng * mq) cell_load(H, t, mq, inv, cw);
    };
    auto prefetch = [&](int g, int p0, WinPrefetch& f) {
        f.h = make_int4(0, 0, 0, 0); f.m = make_double2(0.0, 0.0);
        if (g < g1 && t < (int)(sizeof(WinHdr) / 16)) f.h = reinterpret_cast<const int4*>(P.win_hdr + g)[t];
        if (p0 >= 0 && t >= 32 && t < 32 + 3 * WIN_GP)       // winM is padded by one group
            f.m = reinterpret_cast<const double2*>(P.winM + 6 * (size_t)p0)[t - 32];
    };
    auto store = [&](int hb, int mb, const WinPrefetch& f) {
        if (t < (int)(sizeof(WinHdr) / 16)) reinterpret_cast<int4*>(&s_hdr[hb])[t] = f.h;
        if (t >= 32 && t < 32 + 3 * WIN_GP) reinterpret_cast<double2*>(s_M[mb])[t - 32] = f.m;
    };
    {
        WinPrefetch f;
        prefetch(g0, P.win_hdr[g0].p0, f);
        store(0, 0, f);
        prefetch(g0 + 1, -1, f);
        if (t < (int)(sizeof(WinHdr) / 16)) reinterpret_cast<int4*>(&s_hdr[1])[t] = f.h;
    }
    __syncthreads();
    load_cells(s_hdr[0]);
    int hc = 0, mb = 0;
    for (int g = g0; g < g1; ++g) {
        const int hn = hc == 2 ? 0 : hc + 1, hnn = hn == 2 ? 0 : hn + 1;
        __syncthreads();                                     // Zt is free; header hn and factors mb are in place
        const WinHdr& H = s_hdr[hc];
        const int m6 = 6 * H.m, ng = H.ng;
        const int RT = (m6 + 7) >> 3;
        const int K = 3 * ng, Kp = (K + 3) & ~3;
        // ---- Zt = ([W~ ; Wsh ; g'] M')' from the cells loaded during the previous group's products; the lookup
        //      tables of the epilogue (row / column of the compact product -> offset in the window accumulators)
        {
            const int mq = H.m + 3, ncell = ng * mq;
            const unsigned inv = (0x1000000u + mq - 1) / mq;
            if (t < ncell) cell_put(H, s_M[mb], t, mq, inv, cw);
            for (int idx = t + WIN_TH; idx < ncell; idx += WIN_TH) {                  // unions of more than 14 images
                double2 w[9];
                cell_load(H, idx, mq, inv, w);
                cell_put(H, s_M[mb], idx, mq, inv, w);
            }
            for (int idx = t; idx < (Kp - K) * LDR; idx += WIN_TH) Zt[K * LDR + idx] = 0.0;   // k padding
            if (t < 8 * RT) {                                // row r of the product
                const int a = (t * 43) >> 8, wa = H.wslot[min(a, WIN_MAXW - 1)];
                s_rowTab[t] = t < m6 ? (a << 24) | (((wa * (wa + 1)) >> 1) * 36 + (t - 6 * a) * 6) : -1;
            } else if (t >= 128 && t < 128 + 4 * RT) {       // column pair cc = 2 (t - 128)
                const int cc = 2 * (t - 128), b = (cc * 43) >> 8, wb = H.wslot[min(b, WIN_MAXW - 1)];
                s_colTab[t - 128] = cc < m6 ? (b << 24) | (wb * 36 + (cc - 6 * b)) : (127 << 24);   // 127: never <= a
                s_colSh[t - 128] = cc < m6 ? 6 * wb + (cc - 6 * b) : -1;
            }
        }
        WinPrefetch nxt;
        prefetch(g + 2, g + 1 < g1 ? s_hdr[hn].p0 : -1, nxt);
        __syncthreads();
#ifdef WIN_DEBUG
        for (int i = t; i < Kp * LDR; i += WIN_TH) {
            const double v = Zt[i];
            if (v != v) printf("Zt NaN clu %d g %d k %d row %d (m6 %d ng %d)\n", clu, g, i / LDR, i % LDR, m6, ng);
        }
        for (int i = t; i < 6 * ng; i += WIN_TH) { const double v = s_M[mb][i]; if (v != v) printf("M NaN clu %d g %d i %d\n", clu, g, i); }
        __syncthreads();
#endif
        if (g + 1 < g1) load_cells(s_hdr[hn]);               // in flight during the products
        // ---- tile products, one unit = one A fragment row and up to three column tiles; results straight into
        //      the window accumulators
        const int nUnits = c_winNUnits[RT];
        const int shShift = shRow0 - 8 * RT;                 // virtual -> physical row of the shared tiles
        for (int u = warp; u < nUnits; u += WIN_TH / 32) {
            const unsigned code = c_winUnits[RT][u];
            const int ti = code & 255, tj0 = (code >> 8) & 255, cnt = code >> 16;
            const double* zb = Zt + fk * LDR + fr;
            const double* pa = zb + 8 * ti + (ti >= RT ? shShift : 0);
            const int tj1 = min(tj0 + 1, ti), tj2 = min(tj0 + 2, ti);
            const double* pb0 = zb + 8 * tj0 + (tj0 >= RT ? shShift : 0);
            const double* pb1 = zb + 8 * tj1 + (tj1 >= RT ? shShift : 0);
            const double* pb2 = zb + 8 * tj2 + (tj2 >= RT ? shShift : 0);
            double c[3][2] = {{0.0, 0.0}, {0.0, 0.0}, {0.0, 0.0}};
            if (cnt == 3) win_unit_mma<LDR, 3>(pa, pb0, pb1, pb2, Kp, c);
            else if (cnt == 2) win_unit_mma<LDR, 2>(pa, pb0, pb1, pb2, Kp, c);
            else win_unit_mma<LDR, 1>(pa, pb0, pb1, pb2, Kp, c);
            // epilogue: lane holds C(r, cc), C(r, cc + 1) of every tile (virtual coordinates: camera rows first)
            if (ti < RT) {                                   // camera x camera: block (wa, wb), wb <= wa
                const int rt = s_rowTab[8 * ti + fr];
                if (rt >= 0) {
                    const int a = rt >> 24;
                    double* rowBase = Acc + (rt & 0xffffff);
#pragma unroll
                    for (int n = 0; n < 3; ++n) {
                        if (n < cnt) {
                            const int ct = s_colTab[4 * (tj0 + n) + fk];
                            if ((ct >> 24) <= a) {
                                double2* dst = (double2*)(rowBase + (ct & 0xffffff));
                                double2 v = *dst;
                                v.x += c[n][0]; v.y += c[n][1];
                                *dst = v;
                            }
                        }
                    }
                }
            } else {
                const int s = 8 * (ti - RT) + fr;            // shared row 0..15
#pragma unroll
                for (int n = 0; n < 3; ++n) {
                    if (n < cnt) {
                        const int tj = tj0 + n;
                        const int off = tj < RT ? s_colSh[4 * tj + fk] : 16 * WIN_SHLD + (8 * (tj - RT) + 2 * fk) + s * (16 - WIN_SHLD);
                        if (off >= 0) {                      // AccSS follows AccSh: one base pointer serves both
                            double2* dst = (double2*)(AccSh + s * WIN_SHLD + off);
                            double2 v = *dst;
                            v.x += c[n][0]; v.y += c[n][1];
                            *dst = v;
                        }
                    }
                }
            }
        }
        store(hnn, mb ^ 1, nxt);
        hc = hn; mb ^= 1;
    }
    __syncthreads();
#ifdef WIN_DEBUG
    for (int i = t; i < WIN_ACC + 16 * WIN_SHLD + 256; i += WIN_TH) { const double v = Acc[i]; if (v != v) printf("Acc NaN clu %d i %d\n", clu, i); }
#endif
    // ---- the cluster's window image: blocks (wa >= wb), shared rows, shared x shared
    double* out = P.win_stg + P.clu_stg[clu];
    const int nb = (mw * (mw + 1) / 2) * 36;
    for (int i = 2 * t; i < nb; i += 2 * WIN_TH) *reinterpret_cast<double2*>(out + i) = *reinterpret_cast<const double2*>(Acc + i);
    out += nb;
    for (int i = 2 * t; i < 16 * WIN_SHLD + 256; i += 2 * WIN_TH)
        *reinterpret_cast<double2*>(out + i) = *reinterpret_cast<const double2*>(AccSh + i);
}

// Fixed-order sums of the cluster images into S.  Block ranges of the grid:
//   [0, nbA)          camera-pair blocks: thread = (block, entry), 7 blocks (252 threads) per CTA
//   [nbA, nbA + nbB)  shared-IO x EO rows and the reduced gradient: thread = (image, shared row, EO element), 2 images per CTA
//   [nbA + nbB, ...)  shared x shared: partial sums over WIN_SSPART clusters each
__global__ void __launch_bounds__(256) k_schur_reduce(DevProblem P, int nbA, int nbB) {
    const int t = threadIdx.x;
    if ((int)blockIdx.x < nbA) {
        const int blk = blockIdx.x * 7 + t / 36, e = t % 36;
        if (t >= 252 || blk >= P.nRedBlk) return;
        const int ra = e / 6, cb = e % 6;
        const int iA = P.red_imgA[blk], iB = P.red_imgB[blk];
        const int row = P.eo_s[6 * (size_t)iA + ra], col = P.eo_s[6 * (size_t)iB + cb];
        if (row < 0 || col < 0 || col > row) return;
        const int c0 = P.red_ptr[blk], c1 = P.red_ptr[blk + 1];
        double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
        int c = c0;
        for (; c + 7 < c1; c += 8) {
            const double v0 = P.win_stg[P.red_off[c] + e], v1 = P.win_stg[P.red_off[c + 1] + e];
            const double v2 = P.win_stg[P.red_off[c + 2] + e], v3 = P.win_stg[P.red_off[c + 3] + e];
            const double v4 = P.win_stg[P.red_off[c + 4] + e], v5 = P.win_stg[P.red_off[c + 5] + e];
            const double v6 = P.win_stg[P.red_off[c + 6] + e], v7 = P.win_stg[P.red_off[c + 7] + e];
            s0 += v0; s1 += v1; s2 += v2; s3 += v3; s0 += v4; s1 += v5; s2 += v6; s3 += v7;
        }
        for (; c + 3 < c1; c += 4) {
            s0 += P.win_stg[P.red_off[c] + e]; s1 += P.win_stg[P.red_off[c + 1] + e];
            s2 += P.win_stg[P.red_off[c + 2] + e]; s3 += P.win_stg[P.red_off[c + 3] + e];
        }
        for (; c < c1; ++c) s0 += P.win_stg[P.red_off[c] + e];
        *tc_at(P.T, row, col) -= (s0 + s1) + (s2 + s3);
        return;
    }
    if ((int)blockIdx.x < nbA + nbB) {
        const int img = (blockIdx.x - nbA) * 2 + t / 96, e = t % 96;
        if (t >= 192 || img >= P.nImg) return;
        const int s = e / 6, cb = e % 6;
        if (s > DBAT_NSLOT) return;
        const int col = P.eo_s[6 * (size_t)img + cb];
        if (col < 0) return;
        const int c0 = P.redi_ptr[img], c1 = P.redi_ptr[img + 1];
        double s0 = 0.0, s1 = 0.0;
        int c = c0;
        for (; c + 1 < c1; c += 2) {
            s0 += P.win_stg[P.redi_off[c] + s * WIN_SHLD + cb];
            s1 += P.win_stg[P.redi_off[c + 1] + s * WIN_SHLD + cb];
        }
        if (c < c1) s0 += P.win_stg[P.redi_off[c] + s * WIN_SHLD + cb];
        const double v = s0 + s1;
        if (s < DBAT_NSLOT) {
            const int srow = P.sh_s[s];
            if (srow >= 0) *tc_at(P.T, srow, col) -= v;
        } else {
            P.rhs[col] += v;
        }
        return;
    }
    const int part = blockIdx.x - nbA - nbB;
    const int k0 = part * WIN_SSPART, k1 = min(P.nClu, k0 + WIN_SSPART);
    double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
    int k = k0;
    for (; k + 3 < k1; k += 4) {
        s0 += P.win_stg[P.clu_stg[k + 1] - 256 + t]; s1 += P.win_stg[P.clu_stg[k + 2] - 256 + t];
        s2 += P.win_stg[P.clu_stg[k + 3] - 256 + t]; s3 += P.win_stg[P.clu_stg[k + 4] - 256 + t];
    }
    for (; k < k1; ++k) s0 += P.win_stg[P.clu_stg[k + 1] - 256 + t];
    P.win_ssPart[(size_t)part * 256 + t] = (s0 + s1) + (s2 + s3);
}

// shared x shared block and the shared part of the reduced gradient: sum of the partial tables (+ what the
// per-point kernel of the points with many rays left in shAcc), applied by one CTA
__global__ void __launch_bounds__(256) k_schur_ss_apply(DevProblem P, int nPart, const double* __restrict__ shAcc) {
    const int t = threadIdx.x;
    const int a = t >> 4, b = t & 15;
    if (a >= DBAT_NSLOT || b > DBAT_NSLOT) return;
    double s = shAcc ? shAcc[a * (DBAT_NSLOT + 1) + b] : 0.0;
    const int src = b == DBAT_NSLOT ? DBAT_NSLOT * 16 + a : t;   // only the lower tiles of the table are computed: (a, g) is read as (g, a)
    for (int k = 0; k < nPart; ++k) s += P.win_ssPart[(size_t)k * 256 + src];
    const int row = P.sh_s[a];
    if (row < 0) return;
    if (b < DBAT_NSLOT) {
        const int col = P.sh_s[b];
        if (col < 0 || b > a) return;
        *tc_at(P.T, row, col) -= s;
    } else {
        P.rhs[row] += s;
    }
}

static size_t schur_win_smem(int ldr) {
    return sizeof(double) * ((size_t)(3 * WIN_GP + 2) * ldr + WIN_ACC + 16 * WIN_SHLD + 256);
}
#define WIN_LDR_SMALL win_ldr(8 * ((6 * 12 + 7) / 8) + 16)            // unions of up to 12 images (the default cap)
#define WIN_LDR_LARGE win_ldr(8 * ((6 * WIN_MAXW + 7) / 8) + 16)      // single points with up to WIN_MAXW rays

// S and rhs must hold N_cc + lambda I and -g_c (launch_build_S); shAcc (or null) is added to the shared table
void launch_schur_win(const DevProblem& P, double lambda, const double* shAcc, cudaStream_t st) {
    static thread_local bool init = false;                  // per device: one host thread drives one device
    if (!init) {
        static unsigned int tab[WIN_MAXRT + 1][WIN_MAXUNIT];
        static int cnt[WIN_MAXRT + 1];
        build_units(tab, cnt);
        cudaMemcpyToSymbol(c_winUnits, tab, sizeof(tab));
        cudaMemcpyToSymbol(c_winNUnits, cnt, sizeof(cnt));
        cudaFuncSetAttribute(k_schur_win<WIN_LDR_SMALL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)schur_win_smem(WIN_LDR_SMALL));
        cudaFuncSetAttribute(k_schur_win<WIN_LDR_LARGE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)schur_win_smem(WIN_LDR_LARGE));
        init = true;
    }
    const int nPart = (P.nClu + WIN_SSPART - 1) / WIN_SSPART;
    if (P.nClu > 0) {
        k_point_minv<<<(P.nCand + 255) / 256, 256, 0, st>>>(P, lambda);
        if (P.grpMaxRays <= 12) k_schur_win<WIN_LDR_SMALL><<<P.nClu, WIN_TH, schur_win_smem(WIN_LDR_SMALL), st>>>(P);
        else k_schur_win<WIN_LDR_LARGE><<<P.nClu, WIN_TH, schur_win_smem(WIN_LDR_LARGE), st>>>(P);
        { cudaError_t e = cudaGetLastError(); if (e != cudaSuccess) fprintf(stderr, "dbat: k_schur_win launch failed: %s\n", cudaGetErrorString(e)); }
        const int nbA = (P.nRedBlk + 6) / 7, nbB = (P.nImg + 1) / 2;
        k_schur_reduce<<<nbA + nbB + nPart, 256, 0, st>>>(P, nbA, nbB);
        count_launch(3);
    }
    k_schur_ss_apply<<<1, 256, 0, st>>>(P, nPart, shAcc);
    count_launch();
}
