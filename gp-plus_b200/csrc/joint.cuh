// K4j: the small kernels around the joint predictive covariance and posterior draws (gpp_predict_joint,
// gpp_sample_posterior).  The heavy steps reuse the training-side kernels on the candidate set:
//   K** = cov_tile_kernel (lower tiles, same, identity padding),  Sigma* = K** - U U^T with U = K* L^-T
//   (dgemm_dmma <true,true>, lower tiles), L* = potrf_blocked(Sigma*), draws Y = mu + E L*^T (dgemm_dmma <true,true>).
// Everything here is O(m^2) bookkeeping: diagonal additions, the mirrored upper triangle and the mean rows.
#pragma once
#include <cuda_runtime.h>

namespace gpp {

// diag_add = noise[group] (include_noise) + jitter for the m candidates, 0 on the padding
__global__ void joint_diag_kernel(const int* noise_idx, const double* noise, int n_noise, int include_noise,
                                  double jitter, int m, int mp, double* diag_add) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= mp) return;
    double d = 0.0;
    if (i < m) {
        d = jitter;
        if (include_noise) {
            const int g = noise_idx ? noise_idx[i] : 0;
            if (g >= 0 && g < n_noise) d = noise[g] + jitter;
        }
    }
    diag_add[i] = d;
}

// upper triangle <- transposed lower triangle (32 x 32 blocks through shared memory), so that the returned covariance
// is exactly symmetric; grid (nb, nb), block (32, 8); blocks above the diagonal read the mirrored block below it
__global__ void __launch_bounds__(256) mirror_lower_kernel(double* S, long long ld) {
    __shared__ double t[32][33];
    const int bi = blockIdx.y, bj = blockIdx.x;
    if (bj < bi) return;
    const int tx = threadIdx.x, ty = threadIdx.y;
    if (bj == bi) {
        double* b = S + (long long)bi * 32 * ld + (long long)bj * 32;
        for (int r = ty; r < 32; r += 8)
            if (tx > r) b[(long long)r * ld + tx] = b[(long long)tx * ld + r];
        return;
    }
    const double* src = S + (long long)bj * 32 * ld + (long long)bi * 32;  // lower block (bj, bi)
    for (int r = ty; r < 32; r += 8) t[r][tx] = src[(long long)r * ld + tx];
    __syncthreads();
    double* dst = S + (long long)bi * 32 * ld + (long long)bj * 32;
    for (int r = ty; r < 32; r += 8) dst[(long long)r * ld + tx] = t[tx][r];
}

// strict upper triangle of every diagonal 128-tile <- 0: the leaf writes only the lower triangle of L*, and the draw
// GEMM reads the whole diagonal tile; one CTA per tile
__global__ void __launch_bounds__(256) zero_diag_upper_kernel(double* A, long long ld) {
    double* p = A + (long long)blockIdx.x * 128 * ld + (long long)blockIdx.x * 128;
    for (int idx = threadIdx.x; idx < 128 * 128; idx += blockDim.x) {
        const int r = idx >> 7, c = idx & 127;
        if (c > r) p[(long long)r * ld + c] = 0.0;
    }
}

// every row of Y [rows x mp] <- mu [mp]: C of the draw GEMM, which adds E L*^T with beta = 1
__global__ void fill_rows_kernel(double* Y, const double* mu, long long mp, long long total) {
    for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < total; k += (long long)gridDim.x * blockDim.x)
        Y[k] = mu[k % mp];
}

}  // namespace gpp
