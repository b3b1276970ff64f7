// covstats.cu — report-side consumers of the posterior covariance on the device (SURVEY §8f N2).
//
// Replaces, for the block selectors of bundle_cov, what the reference does on the host after `bundle_cov`:
//   code/misc/corrmat.m:21-47                         R = C ./ (sd sd'), clipped to [-1, 1]
//   code/bundle/private/high_eo_correlations.m, high_op_correlations.m, high_io_correlations.m
//                                                     find(abs(tril(R, -1)) > thres), block by block
//   code/bundle/bundle_result_file.m:92-153           posterior standard deviations = sqrt(diag(C))
// The k x k blocks (EO: 6 x 6 per image, OP: 3 x 3 per point, IO: NC x NC of the shared camera) stay on the device:
// one kernel takes the standard deviations and counts the pairs above the threshold, an exclusive scan (cub) gives
// every block its place in the output, a second kernel writes the pairs in the reference's order (block, then
// column, then row).  Only the standard deviations and the (few) pairs travel to the host.
#include <cub/device/device_scan.cuh>
#include "kernels.cuh"
#include "launch.h"

// blocks: k x k x N, column-major inside a block; cols: k x N, x column of every element or -1 (not estimated)
template <bool EMIT>
__global__ void k_block_corr(const double* __restrict__ blocks, const int* __restrict__ cols, int k, long long N,
                             double thres, double* __restrict__ std_x, int* __restrict__ counts,
                             const long long* __restrict__ offs, long long cap, long long* __restrict__ hitBlock,
                             int* __restrict__ hitRow, int* __restrict__ hitCol, double* __restrict__ hitRho) {
    const long long b = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (b >= N) return;
    const double* C = blocks + (size_t)b * k * k;
    const int* cl = cols + (size_t)b * k;
    if (!EMIT) {
        for (int a = 0; a < k; ++a) if (cl[a] >= 0) std_x[cl[a]] = sqrt(C[a * k + a]);
    }
    long long pos = EMIT ? offs[b] : 0;
    int cnt = 0;
    for (int c = 0; c < k; ++c) {
        if (cl[c] < 0) continue;
        const double sc = sqrt(C[c * k + c]);
        for (int r = c + 1; r < k; ++r) {
            if (cl[r] < 0) continue;
            double rho = C[c * k + r] / sqrt(C[r * k + r]) / sc;      // corrmat.m:38
            rho = fmin(1.0, fmax(-1.0, rho));                          // NaN stays NaN: never a hit
            if (fabs(rho) > thres) {
                if (EMIT && pos < cap) { hitBlock[pos] = b; hitRow[pos] = r; hitCol[pos] = c; hitRho[pos] = rho; }
                ++pos; ++cnt;
            }
        }
    }
    if (!EMIT) counts[b] = cnt;
}
__global__ void k_counts_to_ll(const int* __restrict__ in, long long* __restrict__ out, long long n) {
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i < n) out[i] = in[i];
}

// Returns 0 or a cudaError code; *nHits = number of pairs found (only min(nHits, cap) are written to the host arrays).
int cov_block_stats(const double* d_blocks, const int* d_cols, int k, long long N, double thres, double* d_std_x,
                    long long cap, long long* nHits, long long* h_block, int* h_row, int* h_col, double* h_rho,
                    cudaStream_t st) {
    *nHits = 0;
    if (N <= 0) return 0;
    int* d_cnt = nullptr; long long *d_cnt64 = nullptr, *d_off = nullptr, *d_hb = nullptr; int *d_hr = nullptr, *d_hc = nullptr;
    double* d_hv = nullptr; void* d_tmp = nullptr;
    size_t need = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, need, d_cnt64, d_off, (int)N, st);
    const long long capA = cap > 0 ? cap : 1;
    if (cudaMalloc(&d_cnt, sizeof(int) * N) || cudaMalloc(&d_cnt64, sizeof(long long) * N) || cudaMalloc(&d_off, sizeof(long long) * N) ||
        cudaMalloc(&d_tmp, need ? need : 16) || cudaMalloc(&d_hb, sizeof(long long) * capA) || cudaMalloc(&d_hr, sizeof(int) * capA) ||
        cudaMalloc(&d_hc, sizeof(int) * capA) || cudaMalloc(&d_hv, sizeof(double) * capA)) {
        cudaFree(d_cnt); cudaFree(d_cnt64); cudaFree(d_off); cudaFree(d_tmp); cudaFree(d_hb); cudaFree(d_hr); cudaFree(d_hc); cudaFree(d_hv);
        return (int)cudaErrorMemoryAllocation;
    }
    const int nb = (int)((N + 127) / 128);
    k_block_corr<false><<<nb, 128, 0, st>>>(d_blocks, d_cols, k, N, thres, d_std_x, d_cnt, nullptr, 0, nullptr, nullptr, nullptr, nullptr);
    k_counts_to_ll<<<nb, 128, 0, st>>>(d_cnt, d_cnt64, N);
    cub::DeviceScan::ExclusiveSum(d_tmp, need, d_cnt64, d_off, (int)N, st);
    k_block_corr<true><<<nb, 128, 0, st>>>(d_blocks, d_cols, k, N, thres, nullptr, nullptr, d_off, cap, d_hb, d_hr, d_hc, d_hv);
    count_launch(4);
    long long lastOff = 0; int lastCnt = 0;
    cudaMemcpyAsync(&lastOff, d_off + (N - 1), sizeof(long long), cudaMemcpyDeviceToHost, st);
    cudaMemcpyAsync(&lastCnt, d_cnt + (N - 1), sizeof(int), cudaMemcpyDeviceToHost, st);
    cudaError_t e = cudaGetLastError();                 // launch errors (of these and the caller's earlier kernels)
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e == cudaSuccess) {
        *nHits = lastOff + lastCnt;
        const long long m = *nHits < cap ? *nHits : cap;
        if (m > 0) {
            cudaMemcpyAsync(h_block, d_hb, sizeof(long long) * m, cudaMemcpyDeviceToHost, st);
            cudaMemcpyAsync(h_row, d_hr, sizeof(int) * m, cudaMemcpyDeviceToHost, st);
            cudaMemcpyAsync(h_col, d_hc, sizeof(int) * m, cudaMemcpyDeviceToHost, st);
            cudaMemcpyAsync(h_rho, d_hv, sizeof(double) * m, cudaMemcpyDeviceToHost, st);
            e = cudaStreamSynchronize(st);
        }
    }
    cudaFree(d_cnt); cudaFree(d_cnt64); cudaFree(d_off); cudaFree(d_tmp); cudaFree(d_hb); cudaFree(d_hr); cudaFree(d_hc); cudaFree(d_hv);
    return (int)e;
}

// camera-side blocks from the inverse of the scaled reduced system: out[(i k + b) k + a] = s0^2 C[x2s[cb], x2s[ca]] d_ca d_cb
// (zero rows / columns for elements that are not estimated), cols: k x N x columns
__global__ void k_cam_blocks(const double* __restrict__ C, int ld, const int* __restrict__ x2s, const double* __restrict__ dsc,
                             const int* __restrict__ cols, int k, long long N, double s02, int bad, double* __restrict__ out) {
    const long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (e >= N * k * k) return;
    const long long i = e / (k * k);
    const int q = (int)(e - i * k * k), b = q / k, a = q - b * k;
    const int ca = cols[i * k + a], cb = cols[i * k + b];
    double v = 0.0;
    if (ca >= 0 && cb >= 0) v = bad ? nan("") : s02 * C[(size_t)x2s[cb] * ld + x2s[ca]] * dsc[ca] * dsc[cb];
    out[e] = v;
}
void launch_cam_blocks(const double* C, int ld, const int* x2s, const double* dsc, const int* cols, int k, long long N,
                       double s02, int bad, double* out, cudaStream_t st) {
    const long long n = N * k * k;
    if (n <= 0) return;
    k_cam_blocks<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(C, ld, x2s, dsc, cols, k, N, s02, bad, out);
    count_launch();
}
