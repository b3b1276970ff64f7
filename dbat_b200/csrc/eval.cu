// eval.cu — residual / Jacobian / normal-equation assembly kernels (sm_100a).
//
// Replaces the reference's sparse-Jacobian build and J'*J product
// (code/bundle/cameramodel/multi_res.m:56-315, code/bundle/lsa/levenberg_marquardt.m:76-82)
// with two recompute-instead-of-materialise passes over the observations:
//   k_cam_side   (camera-major order): Gram matrix of the weighted rows [A_io | A_eo | r] per
//                image chunk on the FP64 tensor pipe (DMMA m8n8k4) -> N_io,io, N_io,eo, U_i,
//                g_io, g_eo and r'r in one shot; fixed chunk->image->total summation order,
//                so the result is bit-reproducible.
//   k_point_side (point-major order, one thread per object point): V_j, g_j, the IO x OP
//                cross block and the per-observation EO x OP cross blocks W_o.
// Both are HBM-bound streams (48-52 B read per observation, see DESIGN.md).
#include "kernels.cuh"
#include "launch.h"

// ---------------------------------------------------------------------------------------------
// small utilities
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Deterministic block sum (blockDim.x multiple of 32, <= 1024); result valid in thread 0.
__device__ __forceinline__ double block_sum(double v, double* sm /* >= 32 doubles */) {
    v = warp_sum(v);
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    __syncthreads();
    if (l == 0) sm[w] = v;
    __syncthreads();
    double t = 0.0;
    if (w == 0) {
        t = (l < (int)(blockDim.x >> 5)) ? sm[l] : 0.0;
        t = warp_sum(t);
    }
    return t;
}

// deserialize.m:28-30 on device, in two launches (they sit on the critical path of every evaluation and every trial
// point): one kernel scatters x into the IO / EO / OP value arrays (three lists), one builds the image and IO records.
__global__ void __launch_bounds__(256) k_scatter3(const double* __restrict__ x, ScatterList a, ScatterList b, ScatterList c) {
    int blk = blockIdx.x;
    ScatterList l = a;
    if (blk >= a.nb) { blk -= a.nb; l = b; if (blk >= b.nb) { blk -= b.nb; l = c; } }
    const int k = blk * 256 + threadIdx.x;
    if (k < l.cnt) l.arr[l.dest[k]] = x[l.src[k]];
}
__global__ void __launch_bounds__(128) k_param_setup(DevProblem P, const int* __restrict__ rep, int nIO, int nbImg) {
    if ((int)blockIdx.x < nbImg) {
        const int i = blockIdx.x * 128 + threadIdx.x;
        if (i >= P.nImg) return;
        const double* e = P.EOval + 6 * (size_t)i;
        ImgRec& g = P.img[i];
        g.q0[0] = e[0]; g.q0[1] = e[1]; g.q0[2] = e[2];
        sincos(e[3], &g.sw, &g.cw);
        sincos(e[4], &g.sp, &g.cp);
        sincos(e[5], &g.sk, &g.ck);
        return;
    }
    const int u = (blockIdx.x - nbImg) * 128 + threadIdx.x;
    if (u >= nIO) return;
    const int NC = 5 + P.nK + P.nP;
    const double* c = P.IOval + (size_t)NC * rep[u];
    IORec& r = P.io[u];
    for (int s = 0; s < DBAT_NSLOT; ++s) r.v[s] = 0.0;
    for (int s = 0; s < 5; ++s) r.v[s] = c[s];
    for (int k = 0; k < P.nK; ++k) r.v[DBAT_SLOT_K + k] = c[5 + k];
    for (int k = 0; k < P.nP; ++k) r.v[DBAT_SLOT_P + k] = c[5 + P.nK + k];
}
void launch_set_params(const DevProblem& P, const double* x, ScatterList io, ScatterList eo, ScatterList op,
                       const int* rep, int nIO, cudaStream_t st) {
    io.nb = (io.cnt + 255) / 256; eo.nb = (eo.cnt + 255) / 256; op.nb = (op.cnt + 255) / 256;
    const int nb = io.nb + eo.nb + op.nb;
    if (nb > 0) { k_scatter3<<<nb, 256, 0, st>>>(x, io, eo, op); count_launch(); }
    const int nbImg = (P.nImg + 127) / 128, nbIO = (nIO + 127) / 128;
    if (nbImg + nbIO > 0) { k_param_setup<<<nbImg + nbIO, 128, 0, st>>>(P, rep, nIO, nbImg); count_launch(); }
}

// ---------------------------------------------------------------------------------------------
// camera side: Gram of weighted rows on the FP64 tensor pipe
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void dmma884(double& c0, double& c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}

#ifndef DBAT_EVAL_MINBLOCKS
#define DBAT_EVAL_MINBLOCKS 2
#endif
#define XT_LD 68   // 64 rows + 4: fragment loads (8 cols x 4 rows) hit 32 distinct bank pairs

// One image and one IO record serve a whole chunk: they are staged in shared memory by two TMA bulk copies
// (cp.async.bulk + mbarrier) instead of living in ~56 registers of every thread.
__device__ __forceinline__ void tma_stage(void* sdst, const void* gsrc, unsigned bytes, unsigned long long* bar) {
    const unsigned d = (unsigned)__cvta_generic_to_shared(sdst), b = (unsigned)__cvta_generic_to_shared(bar);
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 :: "r"(d), "l"(gsrc), "r"(bytes), "r"(b) : "memory");
}
template <int MODEL>
__global__ void __launch_bounds__(128, 3) k_cam_side(DevProblem P) {
    extern __shared__ __align__(16) double smem[];
    __shared__ __align__(16) ImgRec s_g;
    __shared__ __align__(16) IORec s_io;
    __shared__ __align__(8) unsigned long long s_bar;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    double* Xt = smem + (size_t)warp * DBAT_GW * XT_LD;    // [GW][XT_LD] per warp
    const Chunk ck = P.chunks[blockIdx.x];
    if (threadIdx.x == 0) {
        const unsigned b = (unsigned)__cvta_generic_to_shared(&s_bar);
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(b) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(b), "r"((unsigned)(sizeof(ImgRec) + sizeof(IORec))) : "memory");
        const ImgRec* gi = P.img + ck.img;
        tma_stage(&s_g, gi, sizeof(ImgRec), &s_bar);
        tma_stage(&s_io, P.io + P.img_io[ck.img], sizeof(IORec), &s_bar);
    }
    __syncthreads();
    {
        const unsigned b = (unsigned)__cvta_generic_to_shared(&s_bar);
        unsigned done = 0;
        while (!done) {
            asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\nselp.u32 %0, 1, 0, p;\n}"
                         : "=r"(done) : "r"(b) : "memory");
        }
    }
    const ImgRec& g = s_g;
    const IORec& io = s_io;

    double acc[DBAT_GTP][2];
#pragma unroll
    for (int t = 0; t < DBAT_GTP; ++t) { acc[t][0] = 0.0; acc[t][1] = 0.0; }
    // padding columns stay zero for the whole kernel
    for (int c = DBAT_COL_R + 1; c < DBAT_GW; ++c) {
        Xt[c * XT_LD + 2 * lane] = 0.0; Xt[c * XT_LD + 2 * lane + 1] = 0.0;
    }

    for (int base = warp * 32; base < ck.count; base += 128) {
        const int k = base + lane;
        ObsJac o;
        double w0 = 0.0, w1 = 0.0;
        const bool valid = k < ck.count;
        if (valid) {
            const int idx = ck.start + k;
            const double2 uv = P.uv_cm[idx];
            const double2 is = P.isig_cm[idx];
            const int j = P.pt_cm[idx];
            const double Q[3] = {P.OPval[3 * (size_t)j], P.OPval[3 * (size_t)j + 1],
                                 P.OPval[3 * (size_t)j + 2]};
            obs_model<MODEL, true, false>(Q, g, io, P.nK, P.nP, uv.x, uv.y, o);
            w0 = is.x; w1 = is.y;
        }
        __syncwarp();
        double2* col;
#pragma unroll
        for (int s = 0; s < DBAT_NSLOT; ++s) {
            col = reinterpret_cast<double2*>(Xt + s * XT_LD) + lane;
            *col = valid ? make_double2(o.dIO[s][0] * w0, o.dIO[s][1] * w1) : make_double2(0.0, 0.0);
        }
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            col = reinterpret_cast<double2*>(Xt + (DBAT_COL_EO + c) * XT_LD) + lane;
            *col = valid ? make_double2(o.dC[0][c] * w0, o.dC[1][c] * w1) : make_double2(0.0, 0.0);
            col = reinterpret_cast<double2*>(Xt + (DBAT_COL_EO + 3 + c) * XT_LD) + lane;
            *col = valid ? make_double2(o.dA[0][c] * w0, o.dA[1][c] * w1) : make_double2(0.0, 0.0);
        }
        col = reinterpret_cast<double2*>(Xt + DBAT_COL_R * XT_LD) + lane;
        *col = valid ? make_double2(o.r[0] * w0, o.r[1] * w1) : make_double2(0.0, 0.0);
        __syncwarp();
        // G(p,q) += X(:,p-tile)' X(:,q-tile): A and B fragments share one load pattern
        const double* fr = Xt + (lane >> 2) * XT_LD + (lane & 3);
#pragma unroll 4
        for (int k0 = 0; k0 < 64; k0 += 4) {
            double f[DBAT_GT];
#pragma unroll
            for (int t = 0; t < DBAT_GT; ++t) f[t] = fr[t * 8 * XT_LD + k0];
            int tp = 0;
#pragma unroll
            for (int p = 0; p < DBAT_GT; ++p)
#pragma unroll
                for (int q = 0; q <= p; ++q) { dmma884(acc[tp][0], acc[tp][1], f[p], f[q]); ++tp; }
        }
    }
    // cross-warp reduction in fixed order, then one partial Gram per chunk
    __syncthreads();
    double* red = smem;                                     // [4][GTP*2][32]
#pragma unroll
    for (int t = 0; t < DBAT_GTP; ++t) {
        red[(warp * DBAT_GTP * 2 + 2 * t) * 32 + lane] = acc[t][0];
        red[(warp * DBAT_GTP * 2 + 2 * t + 1) * 32 + lane] = acc[t][1];
    }
    __syncthreads();
    double* out = P.chunkG + (size_t)blockIdx.x * DBAT_GSZ;
    for (int e = threadIdx.x; e < DBAT_GSZ; e += 128) {
        const int t = e >> 6, l = (e & 63) >> 1, h = e & 1;
        double s = 0.0;
#pragma unroll
        for (int w = 0; w < 4; ++w) s += red[(w * DBAT_GTP * 2 + 2 * t + h) * 32 + l];
        out[e] = s;
    }
}

// ---------------------------------------------------------------------------------------------
// compact camera side: the common self-calibration set - f, principal point, b1, K1-K3, P1-P2 estimated, no skew -
// has 9 IO columns; with the 6 EO columns and the residual that is exactly 16 Gram columns = 2 DMMA tiles = 3 tile
// pairs instead of 6 (half the tensor-pipe work of the 24-wide Gram), and nK / nP are compile-time constants in the
// model.  The chunk Gram leaves the kernel in the same canonical layout (columns of the other slots zero).
// ---------------------------------------------------------------------------------------------
#define CE_MASK 0x0CEFu              // slots f px py b1 | K1 K2 K3 | P1 P2
#define CE_NK 3
#define CE_NP 2
#define CE_NA 9                      // IO columns
#define CE_EO CE_NA                  // first EO column
#define CE_R (CE_NA + 6)             // residual column
__host__ __device__ constexpr int ce_col(int s) { int r = 0; for (int k = 0; k < s; ++k) r += (CE_MASK >> k) & 1; return r; }
static_assert(ce_col(DBAT_NSLOT) == CE_NA && CE_R == 15, "compact column set");

#ifndef CAMC_MINB
#define CAMC_MINB 4                    // 126 registers without spills: four CTAs (16 warps) per SM
#endif
template <int MODEL>
__global__ void __launch_bounds__(128, CAMC_MINB) k_cam_side_c(DevProblem P) {
    extern __shared__ __align__(16) double smem[];
    __shared__ __align__(16) ImgRec s_g;
    __shared__ __align__(16) IORec s_io;
    __shared__ __align__(8) unsigned long long s_bar;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    double* Xt = smem + (size_t)warp * 16 * XT_LD;         // [16][XT_LD] per warp
    const Chunk ck = P.chunks[blockIdx.x];
    if (threadIdx.x == 0) {
        const unsigned b = (unsigned)__cvta_generic_to_shared(&s_bar);
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(b) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(b), "r"((unsigned)(sizeof(ImgRec) + sizeof(IORec))) : "memory");
        tma_stage(&s_g, P.img + ck.img, sizeof(ImgRec), &s_bar);
        tma_stage(&s_io, P.io + P.img_io[ck.img], sizeof(IORec), &s_bar);
    }
    __syncthreads();
    {
        const unsigned b = (unsigned)__cvta_generic_to_shared(&s_bar);
        unsigned done = 0;
        while (!done) {
            asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\nselp.u32 %0, 1, 0, p;\n}"
                         : "=r"(done) : "r"(b) : "memory");
        }
    }
    const ImgRec& g = s_g;
    const IORec& io = s_io;
    double acc[3][2] = {{0.0, 0.0}, {0.0, 0.0}, {0.0, 0.0}};
    for (int base = warp * 32; base < ck.count; base += 128) {
        const int k = base + lane;
        ObsJac o;
        double w0 = 0.0, w1 = 0.0;
        const bool valid = k < ck.count;
        if (valid) {
            const int idx = ck.start + k;
            const double2 uv = P.uv_cm[idx];
            const double2 is = P.isig_cm[idx];
            const int j = P.pt_cm[idx];
            const double Q[3] = {P.OPval[3 * (size_t)j], P.OPval[3 * (size_t)j + 1], P.OPval[3 * (size_t)j + 2]};
            obs_model<MODEL, true, false>(Q, g, io, CE_NK, CE_NP, uv.x, uv.y, o);
            w0 = is.x; w1 = is.y;
        }
        __syncwarp();
        double2* col;
#pragma unroll
        for (int s = 0; s < DBAT_NSLOT; ++s) {
            if ((CE_MASK >> s) & 1) {
                col = reinterpret_cast<double2*>(Xt + ce_col(s) * XT_LD) + lane;
                *col = valid ? make_double2(o.dIO[s][0] * w0, o.dIO[s][1] * w1) : make_double2(0.0, 0.0);
            }
        }
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            col = reinterpret_cast<double2*>(Xt + (CE_EO + c) * XT_LD) + lane;
            *col = valid ? make_double2(o.dC[0][c] * w0, o.dC[1][c] * w1) : make_double2(0.0, 0.0);
            col = reinterpret_cast<double2*>(Xt + (CE_EO + 3 + c) * XT_LD) + lane;
            *col = valid ? make_double2(o.dA[0][c] * w0, o.dA[1][c] * w1) : make_double2(0.0, 0.0);
        }
        col = reinterpret_cast<double2*>(Xt + CE_R * XT_LD) + lane;
        *col = valid ? make_double2(o.r[0] * w0, o.r[1] * w1) : make_double2(0.0, 0.0);
        __syncwarp();
        const double* fr = Xt + (lane >> 2) * XT_LD + (lane & 3);
#pragma unroll 4
        for (int k0 = 0; k0 < 64; k0 += 4) {
            const double f0 = fr[k0], f1 = fr[8 * XT_LD + k0];
            dmma884(acc[0][0], acc[0][1], f0, f0);
            dmma884(acc[1][0], acc[1][1], f1, f0);
            dmma884(acc[2][0], acc[2][1], f1, f1);
        }
    }
    // cross-warp reduction in fixed order, then one partial Gram per chunk in the canonical 24-column layout
    __syncthreads();
    double* red = smem;                                     // [4][3 * 2][32]
#pragma unroll
    for (int t = 0; t < 3; ++t) {
        red[(warp * 6 + 2 * t) * 32 + lane] = acc[t][0];
        red[(warp * 6 + 2 * t + 1) * 32 + lane] = acc[t][1];
    }
    __syncthreads();
    double* out = P.chunkG + (size_t)blockIdx.x * DBAT_GSZ;
    for (int e = threadIdx.x; e < DBAT_GSZ; e += 128) {
        const int tp = e >> 6, l = (e & 63) >> 1, h = e & 1;
        const int p = tp < 1 ? 0 : (tp < 3 ? 1 : 2), q = tp - p * (p + 1) / 2;
        const int R = 8 * p + (l >> 2), C = 8 * q + 2 * (l & 3) + h;                  // canonical Gram entry
        auto cmap = [](int c) -> int {
            if (c < DBAT_NSLOT) return ((CE_MASK >> c) & 1) ? __popc(CE_MASK & ((1u << c) - 1u)) : -1;
            if (c < DBAT_COL_R) return CE_EO + (c - DBAT_COL_EO);
            return c == DBAT_COL_R ? CE_R : -1;
        };
        int a = cmap(R), b = cmap(C);
        double s = 0.0;
        if (a >= 0 && b >= 0) {
            if ((a >> 3) < (b >> 3)) { const int t2 = a; a = b; b = t2; }
            const int tq = (a >> 3) == 0 ? 0 : 1 + (b >> 3);
            const int src = (2 * tq + (b & 1)) * 32 + (a & 7) * 4 + ((b & 7) >> 1);
#pragma unroll
            for (int w = 0; w < 4; ++w) s += red[w * 6 * 32 + src];
        }
        out[e] = s;
    }
}

// per-image Gram = sum of its chunk Grams in chunk order
__global__ void k_cam_reduce(DevProblem P, const int* __restrict__ img_chunk_start) {
    const int i = blockIdx.x;
    const int c0 = img_chunk_start[i], c1 = img_chunk_start[i + 1];
    for (int e = threadIdx.x; e < DBAT_GSZ; e += blockDim.x) {
        double s = 0.0;
        for (int c = c0; c < c1; ++c) s += P.chunkG[(size_t)c * DBAT_GSZ + e];
        P.imgG[(size_t)i * DBAT_GSZ + e] = s;
    }
}

// sum over images in ONE launch: block b owns 64 Gram entries, its 16 thread groups a sixteenth of the images each with
// four loads in flight (the loop is latency-bound); fixed order: bit-reproducible
#define SHR_G 16
__global__ void __launch_bounds__(64 * SHR_G) k_sh_reduce(DevProblem P) {
    __shared__ double part[SHR_G][64];
    const int e = blockIdx.x * 64 + (threadIdx.x & 63), q = threadIdx.x >> 6;
    const int per = (P.nImg + SHR_G - 1) / SHR_G, i0 = min(P.nImg, q * per), i1 = min(P.nImg, i0 + per);
    double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
    int i = i0;
    for (; i + 3 < i1; i += 4) {
        s0 += P.imgG[(size_t)i * DBAT_GSZ + e]; s1 += P.imgG[(size_t)(i + 1) * DBAT_GSZ + e];
        s2 += P.imgG[(size_t)(i + 2) * DBAT_GSZ + e]; s3 += P.imgG[(size_t)(i + 3) * DBAT_GSZ + e];
    }
    for (; i < i1; ++i) s0 += P.imgG[(size_t)i * DBAT_GSZ + e];
    part[q][threadIdx.x & 63] = (s0 + s1) + (s2 + s3);
    __syncthreads();
    if (threadIdx.x < 64) {
        double t = 0.0;
#pragma unroll
        for (int g = 0; g < SHR_G; ++g) t += part[g][threadIdx.x];
        P.shG[e] = t;
    }
}

template <int MODEL>
static void launch_cam_side_t(const DevProblem& P, const int* img_chunk_start, double* tmp,
                              cudaStream_t st) {
    const size_t smem = (size_t)4 * DBAT_GW * XT_LD * sizeof(double);
    static thread_local bool attr_done = false;      // cudaFuncSetAttribute is per device; one host thread drives one device
    if (!attr_done) {
        cudaFuncSetAttribute(k_cam_side<MODEL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        attr_done = true;
    }
    if (P.nChunks > 0) {
        if (P.evalCompact) {
            k_cam_side_c<MODEL><<<P.nChunks, 128, (size_t)4 * 16 * XT_LD * sizeof(double), st>>>(P);
        } else k_cam_side<MODEL><<<P.nChunks, 128, smem, st>>>(P);
    }
    k_cam_reduce<<<P.nImg, 128, 0, st>>>(P, img_chunk_start);
    k_sh_reduce<<<DBAT_GSZ / 64, 64 * SHR_G, 0, st>>>(P);
    (void)tmp;
    count_launch(3);
}

void launch_cam_side(const DevProblem& P, const int* img_chunk_start, double* tmp, cudaStream_t st) {
    switch (P.model) {
        case 0: launch_cam_side_t<0>(P, img_chunk_start, tmp, st); break;
        case 1: launch_cam_side_t<1>(P, img_chunk_start, tmp, st); break;
        case 2: launch_cam_side_t<2>(P, img_chunk_start, tmp, st); break;
        case 3: launch_cam_side_t<3>(P, img_chunk_start, tmp, st); break;
        default: launch_cam_side_t<4>(P, img_chunk_start, tmp, st); break;
    }
}

// ---------------------------------------------------------------------------------------------
// point side: one thread per object point (the points of a list: those with more than DBAT_PSB observations)
// ---------------------------------------------------------------------------------------------
template <int MODEL>
__global__ void __launch_bounds__(128, DBAT_EVAL_MINBLOCKS) k_point_side(DevProblem P, const int* __restrict__ list, int nList) {
    const int jj = blockIdx.x * blockDim.x + threadIdx.x;
    if (jj >= nList) return;
    const int j = list[jj];
    const double Q[3] = {P.OPval[3 * (size_t)j], P.OPval[3 * (size_t)j + 1], P.OPval[3 * (size_t)j + 2]};
    double m[3];
#pragma unroll
    for (int t = 0; t < 3; ++t) m[t] = P.op_col[3 * (size_t)j + t] >= 0 ? 1.0 : 0.0;
    double V[6] = {0, 0, 0, 0, 0, 0}, gq[3] = {0, 0, 0};
    double Wsh[DBAT_NSLOT][3];
#pragma unroll
    for (int s = 0; s < DBAT_NSLOT; ++s) { Wsh[s][0] = 0.0; Wsh[s][1] = 0.0; Wsh[s][2] = 0.0; }
    const int o0 = P.pt_start[j], o1 = P.pt_start[j + 1];
    for (int ob = o0; ob < o1; ++ob) {
        const double2 uv = P.uv_pm[ob];
        const double2 is = P.isig_pm[ob];
        const ImgRec g = P.img[P.img_pm[ob]];
        const IORec io = P.io[g.io];
        ObsJac o;
        obs_model<MODEL, true, true>(Q, g, io, P.nK, P.nP, uv.x, uv.y, o);
        double A[2][3];
#pragma unroll
        for (int t = 0; t < 3; ++t) { A[0][t] = o.dOP[0][t] * is.x * m[t]; A[1][t] = o.dOP[1][t] * is.y * m[t]; }
        const double r0 = o.r[0] * is.x, r1 = o.r[1] * is.y;
        V[0] += A[0][0] * A[0][0] + A[1][0] * A[1][0];
        V[1] += A[0][0] * A[0][1] + A[1][0] * A[1][1];
        V[2] += A[0][0] * A[0][2] + A[1][0] * A[1][2];
        V[3] += A[0][1] * A[0][1] + A[1][1] * A[1][1];
        V[4] += A[0][1] * A[0][2] + A[1][1] * A[1][2];
        V[5] += A[0][2] * A[0][2] + A[1][2] * A[1][2];
#pragma unroll
        for (int t = 0; t < 3; ++t) gq[t] += A[0][t] * r0 + A[1][t] * r1;
#pragma unroll
        for (int s = 0; s < DBAT_NSLOT; ++s) {
            const double a0 = o.dIO[s][0] * is.x, a1 = o.dIO[s][1] * is.y;
#pragma unroll
            for (int t = 0; t < 3; ++t) Wsh[s][t] += a0 * A[0][t] + a1 * A[1][t];
        }
        double* Wo = P.W + (size_t)ob * DBAT_W_STRIDE;
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const double a0 = o.dC[0][c] * is.x, a1 = o.dC[1][c] * is.y;
            const double b0 = o.dA[0][c] * is.x, b1 = o.dA[1][c] * is.y;
#pragma unroll
            for (int t = 0; t < 3; ++t) {
                Wo[c * 3 + t] = a0 * A[0][t] + a1 * A[1][t];
                Wo[(3 + c) * 3 + t] = b0 * A[0][t] + b1 * A[1][t];
            }
        }
    }
    double* rec = P.pt + (size_t)j * DBAT_PT_STRIDE;
#pragma unroll
    for (int k = 0; k < 6; ++k) rec[k] = V[k];
#pragma unroll
    for (int t = 0; t < 3; ++t) rec[6 + t] = gq[t];
    rec[9] = 0.0;
#pragma unroll
    for (int s = 0; s < DBAT_NSLOT; ++s)
#pragma unroll
        for (int t = 0; t < 3; ++t) rec[DBAT_PT_WSH + 3 * s + t] = Wsh[s][t];
}

// prior observations (prior_obs.m:28-65): rows (x_k - prior)/sigma with unit Jacobian.
// OP priors fold into the point records; camera-side priors go to camPriorDiag/G (length nC).
__global__ void k_prior_apply(DevProblem P, const double* __restrict__ x,
                              double* __restrict__ camDiag, double* __restrict__ camG,
                              const int* __restrict__ col2pt /* n-nC: 3*pt+t */) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= P.nPrior) return;
    const int c = P.prior_col[k];
    const double w = P.prior_isig[k];
    const double r = (x[c] - P.prior_val[k]) * w;        // weighted residual
    if (c < P.nC) {
        camDiag[c] += w * w;                             // distinct columns: no race
        camG[c] += w * r;
    } else {
        const int e = col2pt[c - P.nC];
        const int j = e / 3, t = e % 3;
        double* rec = P.pt + (size_t)j * DBAT_PT_STRIDE;
        const int d = (t == 0) ? 0 : (t == 1 ? 3 : 5);
        rec[d] += w * w;
        rec[6 + t] += w * r;
    }
}

// ---------------------------------------------------------------------------------------------
// point side, one thread per OBSERVATION (default).  A block takes a run of whole points with at most DBAT_PSB
// observations.  Phase 1: every thread evaluates its observation once (residual + all partials), writes the
// EO x OP cross block W_o straight to global memory (nine 16-byte stores) and leaves the weighted rows
// [A_op | r | A_io] of its observation in shared memory.  Phase 2: one thread per (point, item) - 14 IO slots, V, g -
// sums the products over the point's observations in image order (deterministic) and writes its piece of the
// point record.  No accumulator lives across observations, so the kernel needs half the registers of the
// one-thread-per-point version and runs at three to four times its occupancy.
// ---------------------------------------------------------------------------------------------
#define PS_ROW 37      // doubles per observation row in shared memory: A_op 6 | r 2 | A_io 28 (+1: odd stride)
template <int MODEL>
__global__ void __launch_bounds__(DBAT_PSB, 3) k_point_side_obs(DevProblem P) {
    __shared__ double rows[DBAT_PSB * PS_ROW];
    const int tid = threadIdx.x;
    const int p0 = P.psb_pt[2 * blockIdx.x], p1 = P.psb_pt[2 * blockIdx.x + 1];
    const int ob0 = P.pt_start[p0], nob = P.pt_start[p1] - ob0;
    if (tid < nob) {
        const int ob = ob0 + tid;
        const int j = P.pt_pm[ob];
        const double2 uv = P.uv_pm[ob];
        const double2 is = P.isig_pm[ob];
        const ImgRec g = P.img[P.img_pm[ob]];
        const IORec io = P.io[g.io];
        const double Q[3] = {P.OPval[3 * (size_t)j], P.OPval[3 * (size_t)j + 1], P.OPval[3 * (size_t)j + 2]};
        ObsJac o;
        obs_model<MODEL, true, true>(Q, g, io, P.nK, P.nP, uv.x, uv.y, o);
        double* row = rows + tid * PS_ROW;
        double A[2][3];
#pragma unroll
        for (int t = 0; t < 3; ++t) {
            const double m = P.op_col[3 * (size_t)j + t] >= 0 ? 1.0 : 0.0;
            A[0][t] = o.dOP[0][t] * is.x * m; A[1][t] = o.dOP[1][t] * is.y * m;
            row[t] = A[0][t]; row[3 + t] = A[1][t];
        }
        row[6] = o.r[0] * is.x; row[7] = o.r[1] * is.y;
#pragma unroll
        for (int s = 0; s < DBAT_NSLOT; ++s) { row[8 + 2 * s] = o.dIO[s][0] * is.x; row[9 + 2 * s] = o.dIO[s][1] * is.y; }
        double w[18];
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const double a0 = o.dC[0][c] * is.x, a1 = o.dC[1][c] * is.y;
            const double b0 = o.dA[0][c] * is.x, b1 = o.dA[1][c] * is.y;
#pragma unroll
            for (int t = 0; t < 3; ++t) {
                w[c * 3 + t] = a0 * A[0][t] + a1 * A[1][t];
                w[(3 + c) * 3 + t] = b0 * A[0][t] + b1 * A[1][t];
            }
        }
        double2* Wo = reinterpret_cast<double2*>(P.W + (size_t)ob * DBAT_W_STRIDE);
#pragma unroll
        for (int q = 0; q < 9; ++q) Wo[q] = make_double2(w[2 * q], w[2 * q + 1]);
    }
    __syncthreads();
    const int nItems = (p1 - p0) * 16;
    for (int item = tid; item < nItems; item += DBAT_PSB) {
        const int j = p0 + (item >> 4), it = item & 15;
        const int r0 = P.pt_start[j] - ob0, r1 = P.pt_start[j + 1] - ob0;
        double* rec = P.pt + (size_t)j * DBAT_PT_STRIDE;
        if (it < DBAT_NSLOT) {                               // IO slot x OP cross block
            double a0 = 0.0, a1 = 0.0, a2 = 0.0;
            for (int r = r0; r < r1; ++r) {
                const double* row = rows + r * PS_ROW;
                const double u0 = row[8 + 2 * it], u1 = row[9 + 2 * it];
                a0 += u0 * row[0] + u1 * row[3]; a1 += u0 * row[1] + u1 * row[4]; a2 += u0 * row[2] + u1 * row[5];
            }
            rec[DBAT_PT_WSH + 3 * it] = a0; rec[DBAT_PT_WSH + 3 * it + 1] = a1; rec[DBAT_PT_WSH + 3 * it + 2] = a2;
        } else if (it == 14) {                               // V_j (upper triangle, row-wise)
            double V[6] = {0, 0, 0, 0, 0, 0};
            for (int r = r0; r < r1; ++r) {
                const double* row = rows + r * PS_ROW;
                V[0] += row[0] * row[0] + row[3] * row[3];
                V[1] += row[0] * row[1] + row[3] * row[4];
                V[2] += row[0] * row[2] + row[3] * row[5];
                V[3] += row[1] * row[1] + row[4] * row[4];
                V[4] += row[1] * row[2] + row[4] * row[5];
                V[5] += row[2] * row[2] + row[5] * row[5];
            }
#pragma unroll
            for (int k = 0; k < 6; ++k) rec[k] = V[k];
        } else {                                             // g_j
            double g0 = 0.0, g1 = 0.0, g2 = 0.0;
            for (int r = r0; r < r1; ++r) {
                const double* row = rows + r * PS_ROW;
                g0 += row[0] * row[6] + row[3] * row[7]; g1 += row[1] * row[6] + row[4] * row[7]; g2 += row[2] * row[6] + row[5] * row[7];
            }
            rec[6] = g0; rec[7] = g1; rec[8] = g2; rec[9] = 0.0;
        }
    }
}

// compact point side (see k_cam_side_c): 9 IO columns, nK / nP compile-time
#define PSC_ROW 27     // A_op 6 | r 2 | A_io x-rows 9 | A_io y-rows 9 (+1: odd stride)
__device__ __constant__ unsigned char c_ceSlot[CE_NA] = {0, 1, 2, 3, 5, 6, 7, 10, 11};
#ifndef PSC_MINB
#define PSC_MINB 5
#endif
template <int MODEL>
__global__ void __launch_bounds__(DBAT_PSB, PSC_MINB) k_point_side_obs_c(DevProblem P) {
    __shared__ __align__(16) double rows[DBAT_PSB * PSC_ROW];
    const int tid = threadIdx.x, lane = tid & 31;
    const int p0 = P.psb_pt[2 * blockIdx.x], p1 = P.psb_pt[2 * blockIdx.x + 1];
    const int ob0 = P.pt_start[p0], nob = P.pt_start[p1] - ob0;
    const bool valid = tid < nob;
    ObsJac o;
    double A[2][3];
    double2 is = make_double2(0.0, 0.0);
    // the warp's own part of `rows` first serves as staging area for its cross blocks: every thread leaves its 144
    // bytes there, then the warp writes the 32 x 144 contiguous bytes of W with fully coalesced 16-byte stores (a
    // per-thread store of W touches 32 different 128-byte lines per instruction)
    double* stage = rows + (tid - lane) * PSC_ROW;
    if (valid) {
        const int ob = ob0 + tid;
        const int j = P.pt_pm[ob];
        const double2 uv = P.uv_pm[ob];
        is = P.isig_pm[ob];
        const ImgRec g = P.img[P.img_pm[ob]];
        const IORec io = P.io[g.io];
        const double Q[3] = {P.OPval[3 * (size_t)j], P.OPval[3 * (size_t)j + 1], P.OPval[3 * (size_t)j + 2]};
        obs_model<MODEL, true, true>(Q, g, io, CE_NK, CE_NP, uv.x, uv.y, o);
#pragma unroll
        for (int t = 0; t < 3; ++t) {
            const double m = P.op_col[3 * (size_t)j + t] >= 0 ? 1.0 : 0.0;
            A[0][t] = o.dOP[0][t] * is.x * m; A[1][t] = o.dOP[1][t] * is.y * m;
        }
        double w[18];
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const double a0 = o.dC[0][c] * is.x, a1 = o.dC[1][c] * is.y;
            const double b0 = o.dA[0][c] * is.x, b1 = o.dA[1][c] * is.y;
#pragma unroll
            for (int t = 0; t < 3; ++t) {
                w[c * 3 + t] = a0 * A[0][t] + a1 * A[1][t];
                w[(3 + c) * 3 + t] = b0 * A[0][t] + b1 * A[1][t];
            }
        }
        double2* sw = reinterpret_cast<double2*>(stage + lane * DBAT_W_STRIDE);
#pragma unroll
        for (int q = 0; q < 9; ++q) sw[q] = make_double2(w[2 * q], w[2 * q + 1]);
    }
    __syncwarp();
    {
        const int nv = min(32, nob - (tid - lane));           // observations of this warp
        double2* Wg = reinterpret_cast<double2*>(P.W + (size_t)(ob0 + tid - lane) * DBAT_W_STRIDE);
        const double2* ss = reinterpret_cast<const double2*>(stage);
#pragma unroll
        for (int q = 0; q < 9; ++q) {
            const int piece = q * 32 + lane;
            if (piece < nv * 9) Wg[piece] = ss[piece];
        }
    }
    __syncwarp();
    if (valid) {
        double* row = rows + tid * PSC_ROW;
#pragma unroll
        for (int t = 0; t < 3; ++t) { row[t] = A[0][t]; row[3 + t] = A[1][t]; }
        row[6] = o.r[0] * is.x; row[7] = o.r[1] * is.y;
#pragma unroll
        for (int s = 0; s < DBAT_NSLOT; ++s) {
            if ((CE_MASK >> s) & 1) { row[8 + ce_col(s)] = o.dIO[s][0] * is.x; row[8 + CE_NA + ce_col(s)] = o.dIO[s][1] * is.y; }
        }
    }
    __syncthreads();
    {
        // Phase 2 on the FP64 tensor pipe: per point the 3 x 13 product  A_op' [A_op | r | A_io]  over its 2 n rows
        // (observation, x/y).  One warp per point; one k-step of m8n8k4 takes two observations; rows 3..7 of the A
        // fragment are zero.  Three shared-memory loads per step instead of ~8 per (item, observation).
        const int warp = tid >> 5;
        const int fm = lane >> 2, fk = lane & 3;             // A: row fm, k fk;  B: k fk, column fm;  C: row fm, columns 2fk, 2fk+1
        const int xy = fk & 1, oo = fk >> 1;
        const int nB = 8 + fm;                               // column of the second tile
        const int offA = 3 * xy + fm;
        const int offB0 = fm < 3 ? 3 * xy + fm : (fm == 3 ? 6 + xy : 8 + CE_NA * xy + (fm - 4));
        const bool b1ok = nB < 4 + CE_NA;
        const int offB1 = 8 + CE_NA * xy + (nB - 4);
        for (int jj = warp; jj < p1 - p0; jj += DBAT_PSB / 32) {
            const int j = p0 + jj;
            const int r0 = P.pt_start[j] - ob0, r1 = P.pt_start[j + 1] - ob0;
            double c00 = 0.0, c01 = 0.0, c10 = 0.0, c11 = 0.0;
            for (int r = r0; r < r1; r += 2) {
                const int ro = r + oo;
                const bool in = ro < r1;
                const double* row = rows + ro * PSC_ROW;
                const double a = (in && fm < 3) ? row[offA] : 0.0;
                const double b0 = in ? row[offB0] : 0.0;
                const double b1 = (in && b1ok) ? row[offB1] : 0.0;
                dmma884(c00, c01, a, b0);
                dmma884(c10, c11, a, b1);
            }
            if (fm < 3) {
                double* rec = P.pt + (size_t)j * DBAT_PT_STRIDE;
                // first tile: columns 0..2 V(fm, .), 3 g(fm), 4..7 IO columns 0..3; second tile: IO columns 4..8
                if (fk == 0) {
                    if (fm == 0) { rec[0] = c00; rec[1] = c01; } else if (fm == 1) rec[3] = c01;
                    rec[DBAT_PT_WSH + 3 * c_ceSlot[4] + fm] = c10; rec[DBAT_PT_WSH + 3 * c_ceSlot[5] + fm] = c11;
                } else if (fk == 1) {
                    rec[fm == 0 ? 2 : (fm == 1 ? 4 : 5)] = c00; rec[6 + fm] = c01;
                    rec[DBAT_PT_WSH + 3 * c_ceSlot[6] + fm] = c10; rec[DBAT_PT_WSH + 3 * c_ceSlot[7] + fm] = c11;
                } else if (fk == 2) {
                    rec[DBAT_PT_WSH + 3 * c_ceSlot[0] + fm] = c00; rec[DBAT_PT_WSH + 3 * c_ceSlot[1] + fm] = c01;
                    rec[DBAT_PT_WSH + 3 * c_ceSlot[8] + fm] = c10;
                } else {
                    rec[DBAT_PT_WSH + 3 * c_ceSlot[2] + fm] = c00; rec[DBAT_PT_WSH + 3 * c_ceSlot[3] + fm] = c01;
                    if (fm == 0) rec[9] = 0.0;
                }
            }
        }
    }
}

template <int MODEL>
static void launch_point_side_t(const DevProblem& P, cudaStream_t st) {
    if (P.nPsb > 0) {
        if (P.evalCompact) k_point_side_obs_c<MODEL><<<P.nPsb, DBAT_PSB, 0, st>>>(P);
        else k_point_side_obs<MODEL><<<P.nPsb, DBAT_PSB, 0, st>>>(P);
        count_launch();
    }
    if (P.nPsbig > 0) { k_point_side<MODEL><<<(P.nPsbig + 127) / 128, 128, 0, st>>>(P, P.psbig, P.nPsbig); count_launch(); }
}
void launch_point_side(const DevProblem& P, cudaStream_t st) {
    if (P.ioGeneral) { launch_point_side_gen(P, st); return; }
    switch (P.model) {
        case 0: launch_point_side_t<0>(P, st); break;
        case 1: launch_point_side_t<1>(P, st); break;
        case 2: launch_point_side_t<2>(P, st); break;
        case 3: launch_point_side_t<3>(P, st); break;
        default: launch_point_side_t<4>(P, st); break;
    }
}
void launch_prior_apply(const DevProblem& P, const double* x, double* camDiag, double* camG,
                        const int* col2pt, bool clear, cudaStream_t st) {
    if (clear || P.nPrior > 0) {             // single rank without prior rows: zeroed at create, nothing ever writes them
        cudaMemsetAsync(camDiag, 0, sizeof(double) * P.nC, st);
        cudaMemsetAsync(camG, 0, sizeof(double) * P.nC, st);
    }
    if (P.nPrior > 0) {
        k_prior_apply<<<(P.nPrior + 127) / 128, 128, 0, st>>>(P, x, camDiag, camG, col2pt);
        count_launch();
    }
}

// ---------------------------------------------------------------------------------------------
// residual only (trial points) and J*p statistics
// ---------------------------------------------------------------------------------------------
#ifndef RES_BLOCK
#define RES_BLOCK 256
#endif
#ifndef RES_MINB
#define RES_MINB 4
#endif
template <int MODEL, bool WRITE>
__global__ void __launch_bounds__(RES_BLOCK, RES_MINB) k_resid(DevProblem P, double* __restrict__ partial,
                                                      double2* __restrict__ r_out, int weighted) {
    __shared__ double sm[32];
    double s = 0.0;
    const int k = blockIdx.x * RES_BLOCK + threadIdx.x;
    if (k < P.nObs) {
        const double2 uv = P.uv_cm[k];
        const double2 is = P.isig_cm[k];
        const int j = P.pt_cm[k];
        const ImgRec g = P.img[P.img_cm[k]];
        const IORec io = P.io[g.io];
        const double Q[3] = {P.OPval[3 * (size_t)j], P.OPval[3 * (size_t)j + 1], P.OPval[3 * (size_t)j + 2]};
        ObsJac o;
        obs_model<MODEL, false, false>(Q, g, io, P.nK, P.nP, uv.x, uv.y, o);
        const double r0 = o.r[0] * is.x, r1 = o.r[1] * is.y;
        s = r0 * r0 + r1 * r1;
        if (WRITE) r_out[k] = weighted ? make_double2(r0, r1) : make_double2(o.r[0], o.r[1]);
    }
    s = block_sum(s, sm);
    if (threadIdx.x == 0) partial[blockIdx.x] = s;
}

// prior rows: residual (x - prior) [* 1/sigma]; sum of squares of the weighted rows
__global__ void k_prior_resid(DevProblem P, const double* __restrict__ x, double* __restrict__ partial,
                              double* __restrict__ r_out, int weighted) {
    __shared__ double sm[32];
    double s = 0.0;
    for (int k = threadIdx.x; k < P.nPrior; k += blockDim.x) {
        const double d = x[P.prior_col[k]] - P.prior_val[k];
        const double r = d * P.prior_isig[k];
        s += r * r;
        if (r_out) r_out[k] = weighted ? r : d;
    }
    s = block_sum(s, sm);
    if (threadIdx.x == 0) partial[0] = s;
}

// out[slot] = sum(partial[0..n)) in a fixed order (single block)
__global__ void k_final_sum(const double* __restrict__ partial, int n, double* __restrict__ out, int slot,
                            int accumulate) {
    __shared__ double sm[32];
    double s = 0.0;
    for (int k = threadIdx.x; k < n; k += blockDim.x) s += partial[k];
    s = block_sum(s, sm);
    if (threadIdx.x == 0) out[slot] = accumulate ? out[slot] + s : s;
}

template <int MODEL>
static void launch_resid_t(const DevProblem& P, const double* x, double* partial, double* scal, int slot,
                           double* r_out, int weighted, cudaStream_t st) {
    const int nb = (P.nObs + RES_BLOCK - 1) / RES_BLOCK;
    if (nb > 0) {
        if (r_out) k_resid<MODEL, true><<<nb, RES_BLOCK, 0, st>>>(P, partial, (double2*)r_out, weighted);
        else       k_resid<MODEL, false><<<nb, RES_BLOCK, 0, st>>>(P, partial, nullptr, weighted);
    }
    k_final_sum<<<1, 1024, 0, st>>>(partial, nb, scal, slot, 0);
    count_launch(2);
    if (P.nPrior > 0) {
        k_prior_resid<<<1, 256, 0, st>>>(P, x, partial, r_out ? r_out + 2 * (size_t)P.nObs : nullptr, weighted);
        k_final_sum<<<1, 32, 0, st>>>(partial, 1, scal, slot, 1);
        count_launch(2);
    }
}
// scal[slot] = r'r (weighted) at the current parameter arrays; optionally writes r (m doubles).
void launch_resid(const DevProblem& P, const double* x, double* partial, double* scal, int slot,
                  double* r_out, int weighted, cudaStream_t st) {
    switch (P.model) {
        case 0: launch_resid_t<0>(P, x, partial, scal, slot, r_out, weighted, st); break;
        case 1: launch_resid_t<1>(P, x, partial, scal, slot, r_out, weighted, st); break;
        case 2: launch_resid_t<2>(P, x, partial, scal, slot, r_out, weighted, st); break;
        case 3: launch_resid_t<3>(P, x, partial, scal, slot, r_out, weighted, st); break;
        default: launch_resid_t<4>(P, x, partial, scal, slot, r_out, weighted, st); break;
    }
}

// scal[slot] = sum of squared weighted prior residuals at x
void launch_prior_rr(const DevProblem& P, const double* x, double* partial, double* scal, int slot, bool clear, cudaStream_t st) {
    if (P.nPrior > 0) {
        k_prior_resid<<<1, 256, 0, st>>>(P, x, partial, nullptr, 1);
        k_final_sum<<<1, 32, 0, st>>>(partial, 1, scal, slot, 0);
        count_launch(2);
    } else if (clear) {                      // single rank without prior rows: zeroed at create and stays zero
        cudaMemsetAsync(scal + slot, 0, sizeof(double), st);
    }
}

// (J p) per observation, recomputed: sums of (Jp)^2 and r.(Jp)
template <int MODEL>
__global__ void __launch_bounds__(RES_BLOCK) k_jp(DevProblem P, const double* __restrict__ p,
                                                   double* __restrict__ partial, int nb) {
    __shared__ double sm[32];
    double s2 = 0.0, sr = 0.0;
    const int k = blockIdx.x * RES_BLOCK + threadIdx.x;
    if (k < P.nObs) {
        const double2 uv = P.uv_cm[k];
        const double2 is = P.isig_cm[k];
        const int j = P.pt_cm[k];
        const int i = P.img_cm[k];
        const ImgRec g = P.img[i];
        const IORec io = P.io[g.io];
        const double Q[3] = {P.OPval[3 * (size_t)j], P.OPval[3 * (size_t)j + 1], P.OPval[3 * (size_t)j + 2]};
        ObsJac o;
        obs_model<MODEL, true, true>(Q, g, io, P.nK, P.nP, uv.x, uv.y, o);
        double j0 = 0.0, j1 = 0.0;
#pragma unroll
        for (int s = 0; s < DBAT_NSLOT; ++s) {
            const int c = P.cam_colx[(size_t)DBAT_NCAM * i + s];          // this image's IO column of the slot
            if (c >= 0) { const double pv = p[c]; j0 += o.dIO[s][0] * pv; j1 += o.dIO[s][1] * pv; }
        }
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            int c = P.eo_col[6 * (size_t)i + a];
            if (c >= 0) { const double pv = p[c]; j0 += o.dC[0][a] * pv; j1 += o.dC[1][a] * pv; }
            c = P.eo_col[6 * (size_t)i + 3 + a];
            if (c >= 0) { const double pv = p[c]; j0 += o.dA[0][a] * pv; j1 += o.dA[1][a] * pv; }
            c = P.op_col[3 * (size_t)j + a];
            if (c >= 0) { const double pv = p[c]; j0 += o.dOP[0][a] * pv; j1 += o.dOP[1][a] * pv; }
        }
        j0 *= is.x; j1 *= is.y;
        s2 = j0 * j0 + j1 * j1;
        sr = (o.r[0] * is.x) * j0 + (o.r[1] * is.y) * j1;
    }
    s2 = block_sum(s2, sm);
    sr = block_sum(sr, sm);
    if (threadIdx.x == 0) { partial[blockIdx.x] = s2; partial[nb + blockIdx.x] = sr; }
}
__global__ void k_prior_jp(DevProblem P, const double* __restrict__ x, const double* __restrict__ p,
                           double* __restrict__ partial) {
    __shared__ double sm[32];
    double s2 = 0.0, sr = 0.0;
    for (int k = threadIdx.x; k < P.nPrior; k += blockDim.x) {
        const int c = P.prior_col[k];
        const double w = P.prior_isig[k];
        const double jp = p[c] * w;
        s2 += jp * jp;
        sr += (x[c] - P.prior_val[k]) * w * jp;
    }
    s2 = block_sum(s2, sm);
    sr = block_sum(sr, sm);
    if (threadIdx.x == 0) { partial[0] = s2; partial[1] = sr; }
}
template <int MODEL>
static void launch_jp_t(const DevProblem& P, const double* x, const double* p, double* partial,
                        double* scal, int slot2, int slotr, cudaStream_t st) {
    const int nb = (P.nObs + RES_BLOCK - 1) / RES_BLOCK;
    if (nb > 0) k_jp<MODEL><<<nb, RES_BLOCK, 0, st>>>(P, p, partial, nb);
    k_final_sum<<<1, 256, 0, st>>>(partial, nb, scal, slot2, 0);
    k_final_sum<<<1, 256, 0, st>>>(partial + nb, nb, scal, slotr, 0);
    count_launch(3);
    if (P.nPrior > 0) {
        k_prior_jp<<<1, 256, 0, st>>>(P, x, p, partial);
        k_final_sum<<<1, 32, 0, st>>>(partial, 1, scal, slot2, 1);
        k_final_sum<<<1, 32, 0, st>>>(partial + 1, 1, scal, slotr, 1);
        count_launch(3);
    }
}
// scal[slot2] = |J p|^2, scal[slotr] = r'(J p) with J, r at the current parameter arrays.
void launch_jp(const DevProblem& P, const double* x, const double* p, double* partial, double* scal,
               int slot2, int slotr, cudaStream_t st) {
    switch (P.model) {
        case 0: launch_jp_t<0>(P, x, p, partial, scal, slot2, slotr, st); break;
        case 1: launch_jp_t<1>(P, x, p, partial, scal, slot2, slotr, st); break;
        case 2: launch_jp_t<2>(P, x, p, partial, scal, slot2, slotr, st); break;
        case 3: launch_jp_t<3>(P, x, p, partial, scal, slot2, slotr, st); break;
        default: launch_jp_t<4>(P, x, p, partial, scal, slot2, slotr, st); break;
    }
}

// ---------------------------------------------------------------------------------------------
// dense per-observation Jacobian blocks for the CSC export (one-off, end of a run)
// layout per observation: [2 rows][NSLOT IO | 3 dC | 3 dA | 3 dOP] = 2 x 23 doubles
// ---------------------------------------------------------------------------------------------
template <int MODEL>
__global__ void __launch_bounds__(128) k_export_jac(DevProblem P, double* __restrict__ out, int weighted) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= P.nObs) return;
    const double2 uv = P.uv_cm[k];
    const double2 is = P.isig_cm[k];
    const int j = P.pt_cm[k];
    const ImgRec g = P.img[P.img_cm[k]];
    const IORec io = P.io[g.io];
    const double Q[3] = {P.OPval[3 * (size_t)j], P.OPval[3 * (size_t)j + 1], P.OPval[3 * (size_t)j + 2]};
    ObsJac o;
    obs_model<MODEL, true, true>(Q, g, io, P.nK, P.nP, uv.x, uv.y, o);
    const double w0 = weighted ? is.x : 1.0, w1 = weighted ? is.y : 1.0;
    const int LD = DBAT_NSLOT + 9;
    double* r0 = out + (size_t)k * 2 * LD;
    double* r1 = r0 + LD;
#pragma unroll
    for (int s = 0; s < DBAT_NSLOT; ++s) { r0[s] = o.dIO[s][0] * w0; r1[s] = o.dIO[s][1] * w1; }
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        r0[DBAT_NSLOT + c] = o.dC[0][c] * w0;      r1[DBAT_NSLOT + c] = o.dC[1][c] * w1;
        r0[DBAT_NSLOT + 3 + c] = o.dA[0][c] * w0;  r1[DBAT_NSLOT + 3 + c] = o.dA[1][c] * w1;
        r0[DBAT_NSLOT + 6 + c] = o.dOP[0][c] * w0; r1[DBAT_NSLOT + 6 + c] = o.dOP[1][c] * w1;
    }
}
// Pattern only (the structural-rank test, levenberg_marquardt.m:126-135): one 64-bit mask per observation, bit
// 23 * row + slot set when that Jacobian entry is non-zero (slots as in k_export_jac) - 8 bytes per observation
// instead of 368, so the exact test runs at any problem size.
template <int MODEL>
__global__ void __launch_bounds__(128) k_export_mask(DevProblem P, unsigned long long* __restrict__ out) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= P.nObs) return;
    const double2 uv = P.uv_cm[k];
    const int j = P.pt_cm[k];
    const ImgRec g = P.img[P.img_cm[k]];
    const IORec io = P.io[g.io];
    const double Q[3] = {P.OPval[3 * (size_t)j], P.OPval[3 * (size_t)j + 1], P.OPval[3 * (size_t)j + 2]};
    ObsJac o;
    obs_model<MODEL, true, true>(Q, g, io, P.nK, P.nP, uv.x, uv.y, o);
    unsigned long long m = 0;
    const int LD = DBAT_NSLOT + 9;
#pragma unroll
    for (int r = 0; r < 2; ++r) {
#pragma unroll
        for (int s = 0; s < DBAT_NSLOT; ++s) if (o.dIO[s][r] != 0.0) m |= 1ull << (LD * r + s);
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            if (o.dC[r][c] != 0.0) m |= 1ull << (LD * r + DBAT_NSLOT + c);
            if (o.dA[r][c] != 0.0) m |= 1ull << (LD * r + DBAT_NSLOT + 3 + c);
            if (o.dOP[r][c] != 0.0) m |= 1ull << (LD * r + DBAT_NSLOT + 6 + c);
        }
    }
    out[k] = m;
}
void launch_export_mask(const DevProblem& P, unsigned long long* out, cudaStream_t st) {
    if (P.nObs <= 0) return;
    const int nb = (P.nObs + 127) / 128;
    switch (P.model) {
        case 0: k_export_mask<0><<<nb, 128, 0, st>>>(P, out); break;
        case 1: k_export_mask<1><<<nb, 128, 0, st>>>(P, out); break;
        case 2: k_export_mask<2><<<nb, 128, 0, st>>>(P, out); break;
        case 3: k_export_mask<3><<<nb, 128, 0, st>>>(P, out); break;
        default: k_export_mask<4><<<nb, 128, 0, st>>>(P, out); break;
    }
    count_launch();
}
void launch_export_jac(const DevProblem& P, double* out, int weighted, cudaStream_t st) {
    if (P.nObs <= 0) return;
    const int nb = (P.nObs + 127) / 128;
    switch (P.model) {
        case 0: k_export_jac<0><<<nb, 128, 0, st>>>(P, out, weighted); break;
        case 1: k_export_jac<1><<<nb, 128, 0, st>>>(P, out, weighted); break;
        case 2: k_export_jac<2><<<nb, 128, 0, st>>>(P, out, weighted); break;
        case 3: k_export_jac<3><<<nb, 128, 0, st>>>(P, out, weighted); break;
        default: k_export_jac<4><<<nb, 128, 0, st>>>(P, out, weighted); break;
    }
    count_launch();
}
