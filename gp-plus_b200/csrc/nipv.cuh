// K4v: batch integrated posterior variance (gpp_nipv_qbatch; botorch's qNegIntegratedPosteriorVariance, whose
// fantasised variance does not depend on the fantasised y, so no rank update of K_y is needed).
//
// With U = K L^-T of any point set, the integration points X_I [M] and a t-batch X_t [q] (all in scaled y units):
//   C_t^T = K(X_t, X_I) - U_t U_I^T                          [q x M], one DMMA GEMM per chunk (engine.cu)
//   G_t   = C_t^T C_t                                        qbatch_syrk_kernel<., true> on the C^T rows
//   A_t   = Sigma_t + diag(noise of the row's group) + j_t I  j_t the first of 0, 1e-8, 1e-7, 1e-6 that factors
//   value = -(1/M) sum_m v_m + (1/M) tr(A_t^-1 G_t)          v_m = sf2 - |U_m|^2 (gpp_ipv_points)
// and for the gradient, the two inputs of the q-batch backward pass:
//   A_bar_t     = -(1/M) A_t^-1 G_t A_t^-1                  (over Sigma_t: the upstream covariance gradient)
//   -A_t^-1 / M                                              (second block buffer: blockdiag(G + G^T) C^T with it is
//                                                             -C_bar^T = -(2/M) A_t^-1 C_t^T)
//
// One CTA per t-batch.  Shared memory holds one q x q matrix (132 KB at q = 128): the factor, then A^-1, then
// A^-1 G; the other operand of each product is read from the t-batch's block in global memory.  Every sum runs in an
// order fixed by the t-batch's own row and column indices, so a t-batch's outputs do not depend on the other
// t-batches of the call or on the chunk split.
#pragma once
#include "qbatch.cuh"

namespace gpp {

constexpr int NV_THREADS = 256;

inline size_t nv_smem_bytes(int q) { return sizeof(double) * ((size_t)q * (q + 1) + q); }

struct NipvArgs {
    double* blk;         // [nb][q][q]: A_t in (Sigma_t + noise); A_bar_t out when grad
    const double* gram;  // [nb][q][q]: G_t = C_t^T C_t
    double* ainv;        // [nb][q][q]: scratch, then -A_t^-1 / M when grad
    int q;
    long long nb;
    double inv_m;        // 1 / M
    double vbar;         // (1/M) sum_m v_m
    int grad;
    double* value;       // [nb]
    double* jitter;      // [nb]
    int* info;           // |= 1: not positive definite after the ladder, |= 2: NaN
};

__global__ void __launch_bounds__(NV_THREADS) nipv_block_kernel(const NipvArgs a) {
    extern __shared__ double nv_sm[];
    __shared__ int s_fail;
    const int q = a.q, tid = threadIdx.x, lq = q + 1;
    double* sM = nv_sm;        // [q][q+1]
    double* sR = sM + q * lq;  // [q] row sums of the trace
    const long long t = blockIdx.x;
    double* blk = a.blk + t * q * q;
    const double* G = a.gram + t * q * q;
    double* Y = a.ainv + t * q * q;

    // L_t in shared memory (the ladder of block_ladder_chol)
    const double jit = block_ladder_chol<NV_THREADS>(blk, q, q, sM, lq, &s_fail);
    if (s_fail) {
        if (tid == 0) {
            atomicOr(a.info, s_fail);
            a.value[t] = 0.0;
            a.jitter[t] = jit;
        }
        return;  // uniform across the CTA
    }
    // Y = L^-1 (lower) into the scratch block, thread j owns column j:
    // Y_ij = (delta_ij - sum_{j<=k<i} L_ik Y_kj) / L_ii
    if (tid < q) {
        const int j = tid;
        for (int i = j; i < q; i++) {
            double v = i == j ? 1.0 : 0.0;
            for (int k = j; k < i; k++) v = fma(-sM[i * lq + k], Y[k * q + j], v);
            Y[i * q + j] = v / sM[i * lq + i];
        }
    }
    __syncthreads();
    // A^-1 = Y^T Y over the shared matrix (the factor is no longer needed), exactly symmetric
    for (int idx = tid; idx < q * q; idx += NV_THREADS) {
        const int i = idx / q, j = idx - i * q;
        if (j > i) continue;
        double v = 0.0;
        for (int k = i; k < q; k++) v = fma(Y[k * q + i], Y[k * q + j], v);
        sM[i * lq + j] = v;
        sM[j * lq + i] = v;
    }
    __syncthreads();
    // tr(A^-1 G) = sum_ij (A^-1)_ij G_ij (both symmetric): row sums in column order, then rows in order
    if (tid < q) {
        double r = 0.0;
        for (int j = 0; j < q; j++) r = fma(sM[tid * lq + j], G[tid * q + j], r);
        sR[tid] = r;
    }
    __syncthreads();
    if (tid == 0) {
        double tr = 0.0;
        for (int i = 0; i < q; i++) tr += sR[i];
        const double v = tr * a.inv_m - a.vbar;
        if (isnan(v)) atomicOr(a.info, 2);
        a.value[t] = v;
        a.jitter[t] = jit;
    }
    if (!a.grad) return;
    // H = A^-1 G into the scratch block (Y is no longer needed)
    for (int idx = tid; idx < q * q; idx += NV_THREADS) {
        const int i = idx / q, j = idx - i * q;
        double v = 0.0;
        for (int k = 0; k < q; k++) v = fma(sM[i * lq + k], G[k * q + j], v);
        Y[idx] = v;
    }
    __syncthreads();
    // A_bar = -(1/M) H A^-1 over A_t
    for (int idx = tid; idx < q * q; idx += NV_THREADS) {
        const int i = idx / q, j = idx - i * q;
        double v = 0.0;
        for (int k = 0; k < q; k++) v = fma(Y[i * q + k], sM[k * lq + j], v);
        blk[idx] = -a.inv_m * v;
    }
    __syncthreads();
    for (int idx = tid; idx < q * q; idx += NV_THREADS) {
        const int i = idx / q, j = idx - i * q;
        Y[idx] = -a.inv_m * sM[i * lq + j];
    }
}

inline cudaError_t launch_nipv_block(const NipvArgs& a, cudaStream_t st) {
    if (a.nb <= 0) return cudaSuccess;
    count_launch();
    const size_t smem = nv_smem_bytes(a.q);
    cudaError_t e = cudaFuncSetAttribute(nipv_block_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    nipv_block_kernel<<<(unsigned)a.nb, NV_THREADS, smem, st>>>(a);
    return cudaGetLastError();
}

}  // namespace gpp
