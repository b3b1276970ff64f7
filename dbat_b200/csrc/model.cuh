// model.cuh — per-observation collinearity residual with Brown lens distortion and its
// analytic Jacobian blocks, all in registers (one thread = one observation).
//
// Closed forms of the reference's building-block chain (code/bundle/cameramodel/):
//   eulerrotmat.m:81,100-124 (M=R1R2R3, dM), eulerpinhole2.m:50-108, world2cam.m:45-84,
//   pinhole.m:39-67, scale2.m:41, aniscale2.m:43, aniscale2b.m:41, xlat2.m:41,
//   affine2.m:42, skew.m:41, brown_dist.m:50-91, brown_rad.m:46-95, brown_tang.m:58-138,
//   rad_scale.m:43-77, tang_scale.m:43-89, res_euler_brown_{0,1,2,3}.m (models 2..5).
// FP64 throughout.  Powers r^(2k) are formed by repeated multiplication (the reference's
// power_vec.m:42 uses pow); the difference is below 1 ulp per term and far inside the
// 1e-12 residual tolerance.
#pragma once
#include <cuda_runtime.h>

#define DBAT_KMAX 5                       // max radial coefficients
#define DBAT_PMAX 4                       // max tangential coefficients
#define DBAT_NSLOT (5 + DBAT_KMAX + DBAT_PMAX)   // IO slots: f,px,py,b1,b2,K[KMAX],P[PMAX]
#define DBAT_SLOT_K 5
#define DBAT_SLOT_P (5 + DBAT_KMAX)

// Per-image record rebuilt from x before every evaluation (k_param_setup, eval.cu).
struct __align__(16) ImgRec {
    double sw, cw, sp, cp, sk, ck;        // sin/cos of omega, phi, kappa
    double q0[3];                         // camera centre
    double sz;                            // pixel size x (pxSize(1,img), multi_res.m:138)
    int    io;                            // index of this image's IO record
    int    pad_;
    double szy;                           // pixel size y: = sz for models 2-5, pxSize(2,.) for the legacy models
};
static_assert(sizeof(ImgRec) == 96, "ImgRec layout");

// One IO record in SLOT layout (unpackio.m:4-8 order, K/P padded to KMAX/PMAX).
struct __align__(16) IORec {
    double v[DBAT_NSLOT + (DBAT_NSLOT & 1)];
};

struct ObsJac {
    double r[2];                          // residual v = lhs - l   (unweighted, mm)
    double dOP[2][3];                     // d v / d Q
    double dC[2][3];                      // d v / d q0
    double dA[2][3];                      // d v / d (omega,phi,kappa)
    double dIO[DBAT_NSLOT][2];            // d v / d IO slot
};

__device__ __forceinline__ void rotmat(const ImgRec& g, double M[3][3]) {
    // M = R1(omega) R2(phi) R3(kappa), eulerrotmat.m:81 (seq 123, moving axes)
    M[0][0] = g.cp * g.ck;                 M[0][1] = -g.cp * g.sk;                M[0][2] = g.sp;
    M[1][0] = g.cw * g.sk + g.sw * g.sp * g.ck;
    M[1][1] = g.cw * g.ck - g.sw * g.sp * g.sk;
    M[1][2] = -g.sw * g.cp;
    M[2][0] = g.sw * g.sk - g.cw * g.sp * g.ck;
    M[2][1] = g.sw * g.ck + g.cw * g.sp * g.sk;
    M[2][2] = g.cw * g.cp;
}

// Brown distortion of point a with coefficients Kt=-K, Pt=-P (brown_dist.m:50-58).
// Returns l, D = dl/da (2x2), r2 powers pw[k]=r2^(k+1).
template <bool JAC>
__device__ __forceinline__ void brown(const double a[2], const double* Kt, int nK,
                                      const double* Pt, int nP, double l[2], double D[2][2],
                                      double pw[DBAT_KMAX > DBAT_PMAX ? DBAT_KMAX : DBAT_PMAX],
                                      double ts[2], double& onePlusRsP) {
    const double r2 = a[0] * a[0] + a[1] * a[1];
    constexpr int NPW = DBAT_KMAX > DBAT_PMAX ? DBAT_KMAX : DBAT_PMAX;
    double p = 1.0;
#pragma unroll
    for (int k = 0; k < NPW; ++k) { p *= r2; pw[k] = p; }
    double rad = 0.0, drad = 0.0;          // rad_scale.m:43-51,75
    {
        double pm1 = 1.0;                  // r2^(k)
#pragma unroll
        for (int k = 0; k < DBAT_KMAX; ++k) {
            if (k < nK) { rad += Kt[k] * pw[k]; drad += (k + 1) * Kt[k] * pm1; }
            pm1 = pw[k];
        }
    }
    double p0 = 0.0, p1 = 0.0;
    if (nP >= 2) { p0 = Pt[0]; p1 = Pt[1]; }
    const double pTu = p0 * a[0] + p1 * a[1];  // tang_scale.m:43-45
    ts[0] = p0 * r2 + 2.0 * pTu * a[0];
    ts[1] = p1 * r2 + 2.0 * pTu * a[1];
    double rsP = 0.0, drsP = 0.0;          // brown_tang.m:60-70 (P(3:end))
    {
        double pm1 = 1.0;
#pragma unroll
        for (int k = 0; k < DBAT_PMAX - 2; ++k) {
            if (k + 2 < nP) { rsP += Pt[k + 2] * pw[k]; drsP += (k + 1) * Pt[k + 2] * pm1; }
            pm1 = pw[k];
        }
    }
    onePlusRsP = 1.0 + rsP;
    l[0] = a[0] + a[0] * rad + ts[0] * onePlusRsP;
    l[1] = a[1] + a[1] * rad + ts[1] * onePlusRsP;
    if (JAC) {
        // brown_rad.m:82-93 : rs*I + a*(2*drad)*a' ; tang_scale.m:76-87 ; brown_tang.m:108-134
        const double g2 = 2.0 * drad;
        const double t00 = 2.0 * (2.0 * p0 * a[0] + pTu);
        const double t01 = 2.0 * (p0 * a[1] + p1 * a[0]);
        const double t11 = 2.0 * (2.0 * p1 * a[1] + pTu);
        const double h2 = 2.0 * drsP;
        D[0][0] = 1.0 + rad + g2 * a[0] * a[0] + t00 * onePlusRsP + ts[0] * h2 * a[0];
        D[0][1] = g2 * a[0] * a[1] + t01 * onePlusRsP + ts[0] * h2 * a[1];
        D[1][0] = g2 * a[1] * a[0] + t01 * onePlusRsP + ts[1] * h2 * a[0];
        D[1][1] = 1.0 + rad + g2 * a[1] * a[1] + t11 * onePlusRsP + ts[1] * h2 * a[1];
    }
}

// MODEL = distModel-2 (res_euler_brown_<MODEL>.m) for models 2..5; legacy model 1 is
// arithmetically identical to model 2 (brown_euler_cam4.m:46-59: v = pp - f*h - (m - ld(m-pp)))
// and runs as MODEL 0; MODEL 4 is the forward (computer-vision) model -1
// (brown_euler_cam4.m:193-208,238-281; cammodel/browndist.m:103-253):
//   v = pp + w + ld(w) - m,  w = -f*h,  distortion evaluated at the projected point.
// JAC_CAM: also IO/EO partials; JAC_OP: also OP partials.  Residual rows are x then y, in mm,
// UNWEIGHTED.
template <int MODEL, bool JAC_CAM, bool JAC_OP>
__device__ __forceinline__ void obs_model(const double Q[3], const ImgRec& g, const IORec& io,
                                          int nK, int nP, double ux, double uy, ObsJac& o) {
    double M[3][3];
    rotmat(g, M);
    const double X0 = Q[0] - g.q0[0], X1 = Q[1] - g.q0[1], X2 = Q[2] - g.q0[2];   // xlat3.m:41
    const double q0 = M[0][0] * X0 + M[1][0] * X1 + M[2][0] * X2;                 // M' X
    const double q1 = M[0][1] * X0 + M[1][1] * X1 + M[2][1] * X2;
    const double q2 = M[0][2] * X0 + M[1][2] * X1 + M[2][2] * X2;
    const double zi = 1.0 / q2;
    const double h0 = q0 * zi, h1 = q1 * zi;                                       // pinhole.m:39
    const double f = io.v[0];
    const double lhs0 = -f * h0, lhs1 = -f * h1;                                   // eulerpinhole2 with -f

    // image side
    const double y0 = g.sz * ux, y1 = -g.szy * uy;                                 // scale2, aniscale2([1;-1])
    const double px = io.v[1], py = io.v[2], b1 = io.v[3], b2 = io.v[4];
    double Kt[DBAT_KMAX], Pt[DBAT_PMAX];
    const double sgn = (MODEL == 4) ? 1.0 : -1.0;      // backward models distort with -K,-P
#pragma unroll
    for (int k = 0; k < DBAT_KMAX; ++k) Kt[k] = sgn * io.v[DBAT_SLOT_K + k];
#pragma unroll
    for (int k = 0; k < DBAT_PMAX; ++k) Pt[k] = sgn * io.v[DBAT_SLOT_P + k];
    constexpr int NPW = DBAT_KMAX > DBAT_PMAX ? DBAT_KMAX : DBAT_PMAX;
    double a[2], l[2], D[2][2], pw[NPW], ts[2], opr;
    double x0, x1;
    if (MODEL == 3) { x0 = (1.0 + b1) * y0 - px; x1 = y1 - py; }                   // aniscale2b then xlat2
    else            { x0 = y0 - px;              x1 = y1 - py; }
    if (MODEL == 1)      { a[0] = (1.0 + b1) * x0 + b2 * x1; a[1] = x1; }          // affine2 before brown
    else if (MODEL == 4) { a[0] = lhs0; a[1] = lhs1; }                             // forward: distort the projection
    else                 { a[0] = x0; a[1] = x1; }
    brown<(JAC_CAM || JAC_OP)>(a, Kt, nK, Pt, nP, l, D, pw, ts, opr);
    double rhs0, rhs1;
    if (MODEL == 2)      { rhs0 = (1.0 + b1) * l[0] + b2 * l[1]; rhs1 = l[1]; }    // affine2 after brown
    else if (MODEL == 3) { rhs0 = l[0] + b2 * l[1];              rhs1 = l[1]; }    // skew after brown
    else                 { rhs0 = l[0];                          rhs1 = l[1]; }
    if (MODEL == 4) { o.r[0] = px + l[0] - y0; o.r[1] = py + l[1] - y1; }          // ptDist - m
    else            { o.r[0] = lhs0 - rhs0;    o.r[1] = lhs1 - rhs1; }

    if (JAC_CAM || JAC_OP) {
        // H = dpinhole = zi*[1 0 -h0; 0 1 -h1]; G = -f*H*M'  (2x3) = d lhs / dQ
        double G[2][3];
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            // (H M')[0][c] = zi*(M[c][0] - h0*M[c][2])
            const double g0 = -f * zi * (M[c][0] - h0 * M[c][2]);
            const double g1 = -f * zi * (M[c][1] - h1 * M[c][2]);
            if (MODEL == 4) { G[0][c] = D[0][0] * g0 + D[0][1] * g1; G[1][c] = D[1][0] * g0 + D[1][1] * g1; }   // (I+G_ld) dxy
            else            { G[0][c] = g0; G[1][c] = g1; }
        }
        if (JAC_OP) {
#pragma unroll
            for (int c = 0; c < 3; ++c) { o.dOP[0][c] = G[0][c]; o.dOP[1][c] = G[1][c]; }
        }
        if (JAC_CAM) {
#pragma unroll
            for (int c = 0; c < 3; ++c) { o.dC[0][c] = -G[0][c]; o.dC[1][c] = -G[1][c]; }
            // angles: d lhs/d alpha = -f*H*(dM_alpha)' X
            // omega: (P1 M)' X = -M[2][c]*X1 + M[1][c]*X2
            // phi  : (R1 dR2 R3)' X ; kappa: (M P3)' X = [q1, -q0, 0]
            double w[3][3];
#pragma unroll
            for (int c = 0; c < 3; ++c) w[0][c] = -M[2][c] * X1 + M[1][c] * X2;
            {
                const double d00 = -g.sp * g.ck, d01 = g.sp * g.sk, d02 = g.cp;
                const double d10 = g.sw * g.cp * g.ck, d11 = -g.sw * g.cp * g.sk, d12 = g.sw * g.sp;
                const double d20 = -g.cw * g.cp * g.ck, d21 = g.cw * g.cp * g.sk, d22 = -g.cw * g.sp;
                w[1][0] = d00 * X0 + d10 * X1 + d20 * X2;
                w[1][1] = d01 * X0 + d11 * X1 + d21 * X2;
                w[1][2] = d02 * X0 + d12 * X1 + d22 * X2;
            }
            w[2][0] = q1; w[2][1] = -q0; w[2][2] = 0.0;
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                const double g0 = -f * zi * (w[k][0] - h0 * w[k][2]);
                const double g1 = -f * zi * (w[k][1] - h1 * w[k][2]);
                if (MODEL == 4) { o.dA[0][k] = D[0][0] * g0 + D[0][1] * g1; o.dA[1][k] = D[1][0] * g0 + D[1][1] * g1; }
                else            { o.dA[0][k] = g0; o.dA[1][k] = g1; }
            }
            // IO partials
#pragma unroll
            for (int s = 0; s < DBAT_NSLOT; ++s) { o.dIO[s][0] = 0.0; o.dIO[s][1] = 0.0; }
            if (MODEL == 4) {                                                       // (I+G_ld) * (-h), dv/dpp = I
                o.dIO[0][0] = -(D[0][0] * h0 + D[0][1] * h1); o.dIO[0][1] = -(D[1][0] * h0 + D[1][1] * h1);
            } else {
                o.dIO[0][0] = -h0; o.dIO[0][1] = -h1;                              // dv/df = -h
            }
            // E = d rhs / d a-chain; model specific outer 2x2 "T" applied after brown
            double T00 = 1.0, T01 = 0.0;                                           // T = [T00 T01; 0 1]
            if (MODEL == 2) { T00 = 1.0 + b1; T01 = b2; }
            if (MODEL == 3) { T01 = b2; }
            // TD = T*D
            const double TD00 = T00 * D[0][0] + T01 * D[1][0], TD01 = T00 * D[0][1] + T01 * D[1][1];
            const double TD10 = D[1][0], TD11 = D[1][1];
            // dv/du0 = T*D*A  (A = affine before brown for model 3(=MODEL 1), else I)
            if (MODEL == 4) {
                o.dIO[1][0] = 1.0; o.dIO[2][1] = 1.0;
            } else if (MODEL == 1) {
                o.dIO[1][0] = TD00 * (1.0 + b1); o.dIO[1][1] = TD10 * (1.0 + b1);
                o.dIO[2][0] = TD00 * b2 + TD01;  o.dIO[2][1] = TD10 * b2 + TD11;
            } else {
                o.dIO[1][0] = TD00; o.dIO[1][1] = TD10;
                o.dIO[2][0] = TD01; o.dIO[2][1] = TD11;
            }
            // dv/dK_k = T * a * r2^k   (brown_rad.m:74-78)
#pragma unroll
            for (int k = 0; k < DBAT_KMAX; ++k) {
                if (k < nK) {
                    const double v0 = a[0] * pw[k], v1 = a[1] * pw[k];
                    o.dIO[DBAT_SLOT_K + k][0] = T00 * v0 + T01 * v1;
                    o.dIO[DBAT_SLOT_K + k][1] = v1;
                }
            }
            // dv/dP (tang_scale.m:66-73, brown_tang.m:93-103)
            if (nP >= 2) {
                const double r2 = a[0] * a[0] + a[1] * a[1];
                const double e00 = (r2 + 2.0 * a[0] * a[0]) * opr, e01 = 2.0 * a[0] * a[1] * opr;
                const double e11 = (r2 + 2.0 * a[1] * a[1]) * opr;
                o.dIO[DBAT_SLOT_P + 0][0] = T00 * e00 + T01 * e01; o.dIO[DBAT_SLOT_P + 0][1] = e01;
                o.dIO[DBAT_SLOT_P + 1][0] = T00 * e01 + T01 * e11; o.dIO[DBAT_SLOT_P + 1][1] = e11;
#pragma unroll
                for (int k = 0; k < DBAT_PMAX - 2; ++k) {
                    if (k + 2 < nP) {
                        const double v0 = ts[0] * pw[k], v1 = ts[1] * pw[k];
                        o.dIO[DBAT_SLOT_P + 2 + k][0] = T00 * v0 + T01 * v1;
                        o.dIO[DBAT_SLOT_P + 2 + k][1] = v1;
                    }
                }
            }
            // dv/db
            if (MODEL == 1) {            // -D*[x0 x1; 0 0]   (res_euler_brown_1.m:177)
                o.dIO[3][0] = -D[0][0] * x0; o.dIO[3][1] = -D[1][0] * x0;
                o.dIO[4][0] = -D[0][0] * x1; o.dIO[4][1] = -D[1][0] * x1;
            } else if (MODEL == 2) {     // -[l0 l1; 0 0]
                o.dIO[3][0] = -l[0]; o.dIO[4][0] = -l[1];
            } else if (MODEL == 3) {     // -[SK*D*[y0;0], [l1;0]]
                o.dIO[3][0] = -TD00 * y0; o.dIO[3][1] = -TD10 * y0;
                o.dIO[4][0] = -l[1];
            }
        }
    }
}
