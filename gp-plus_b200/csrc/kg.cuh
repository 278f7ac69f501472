// K4k: one-shot knowledge gradient on the t-batch posteriors of qbatch.cuh (gpp_kg_qbatch; botorch's
// qKnowledgeGradient.forward with the PosteriorMean value function and current_value = None, on the
// X_actual_and_fantasies layout of _split_fantasy_points).
//
// Each t-batch t holds q_tot = q + F rows: the q actual points, then the F fantasy solutions.  One CTA per t-batch,
// after qbatch_syrk_kernel has written its q_tot x q_tot block Sigma (with the observation noise of every row):
//   L_t = chol(Sigma[0:q, 0:q] + j_t I)      j_t the first rung of 0, 1e-8, 1e-7, 1e-6 that factors (block_ladder_chol)
//   w_f = L_t^-1 c_f,  c_f = Sigma[0:q, q+f]  posterior cross-covariance of the actual points and fantasy solution f
//   v_t = (1/F) sum_f sigma (mu[q+f] + w_f . e_f)   (sigma = +1 / -1 to maximise / minimise, e_f [q] row f of the
//                                                    base samples, shared by every t-batch)
// Each term is the posterior mean at fantasy solution f of the model that also observed X_t at mu[0:q] + L_t e_f.
// For the gradient, with v_f = L_t^-T e_f, the two inputs of the q-batch backward:
//   mu_bar[q+f] = sigma / F, mu_bar of the actual rows 0
//   Sigma_bar[i, q+f] = Sigma_bar[q+f, i] = sigma v_f[i] / (2F)   (the cross-covariance gradient, split evenly over
//                                                                   both triangles so the block stays symmetric)
//   L_bar = -(sigma / F) sum_f v_f w_f^T, then Sigma_bar[0:q, 0:q] by block_chol_adjoint; the fantasy block is 0
// Sigma_bar overwrites Sigma and mu_bar goes to the chunk's mean-gradient rows.
//
// Thread f < F owns fantasy f (its two triangular solves and its term); every sum runs in an order fixed by the
// t-batch's own row, column and fantasy indices, so a t-batch's outputs do not depend on the other t-batches of the
// call or on the chunk split.
#pragma once
#include "qbatch.cuh"

namespace gpp {

constexpr int KG_THREADS = 256;

// doubles of dynamic shared memory: L [q x (q+1)], w_f and v_f [F x (q|1)] each, the F terms
inline size_t kg_smem_bytes(int q, int nf) {
    return sizeof(double) * ((size_t)q * (q + 1) + 2 * (size_t)nf * (q | 1) + nf);
}

struct KgArgs {
    double* blk;       // [nb][q_tot][q_tot]: Sigma_t in; Sigma_bar_t out when grad
    const double* mu;  // chunk means in the tile layout (predict_finish_kernel)
    double* gm;        // chunk mean gradients in the tile layout (grad)
    const double* E;   // [F][q] base samples
    int q, nf, qpt;    // actual rows, fantasies, t-batches per 128-row tile
    long long nb;      // t-batches in the chunk
    double sgn;        // +1 maximise, -1 minimise
    int grad;
    double* value;     // [nb]
    double* jitter;    // [nb]
    int* info;         // |= 1: a t-batch is not positive definite after the ladder, |= 2: NaN
};

__global__ void __launch_bounds__(KG_THREADS) kg_block_kernel(const KgArgs a) {
    extern __shared__ double kg_sm[];
    __shared__ int s_fail;
    const int q = a.q, nf = a.nf, qt = q + nf, tid = threadIdx.x, lq = q + 1, ld = q | 1;
    double* sL = kg_sm;           // [q][q+1]
    double* sW = sL + q * lq;     // [F][ld] w_f
    double* sV = sW + nf * ld;    // [F][ld] v_f
    double* sT = sV + nf * ld;    // [F] terms
    const long long t = blockIdx.x;
    const long long r0 = (t / a.qpt) * CT + (t % a.qpt) * qt;  // first row of t in the tile layout
    double* blk = a.blk + t * qt * qt;

    for (int i = tid; i < qt; i += KG_THREADS)
        if (isnan(a.mu[r0 + i])) atomicOr(a.info, 2);
    const double jit = block_ladder_chol<KG_THREADS>(blk, q, qt, sL, lq, &s_fail);
    if (s_fail) {
        if (tid == 0) {
            atomicOr(a.info, s_fail);
            a.value[t] = 0.0;
            a.jitter[t] = jit;
        }
        return;  // uniform across the CTA
    }
    bool nan_seen = false;
    for (int f = tid; f < nf; f += KG_THREADS) {
        const double* e = a.E + (size_t)f * q;
        double* w = sW + f * ld;
        double dot = 0.0;
        for (int i = 0; i < q; i++) {  // w_f = L^-1 c_f, forward in i
            const double* Li = sL + i * lq;
            double v = blk[(size_t)i * qt + q + f];
            for (int k = 0; k < i; k++) v = fma(-Li[k], w[k], v);
            w[i] = v / Li[i];
            dot = fma(w[i], e[i], dot);
        }
        const double term = a.sgn * (a.mu[r0 + q + f] + dot);
        nan_seen |= isnan(term);
        sT[f] = term;
        if (a.grad) {
            double* v = sV + f * ld;
            for (int i = q - 1; i >= 0; i--) {  // v_f = L^-T e_f, backward in i
                double s = e[i];
                for (int k = i + 1; k < q; k++) s = fma(-sL[k * lq + i], v[k], s);
                v[i] = s / sL[i * lq + i];
            }
        }
    }
    if (nan_seen) atomicOr(a.info, 2);
    __syncthreads();
    const double inv_f = 1.0 / (double)nf;
    if (tid == 0) {
        double s = 0.0;
        for (int f = 0; f < nf; f++) s += sT[f];
        a.value[t] = s * inv_f;
        a.jitter[t] = jit;
    }
    if (!a.grad) return;
    const double gs = a.sgn * inv_f;
    for (int i = tid; i < qt; i += KG_THREADS) a.gm[r0 + i] = i < q ? 0.0 : gs;
    // the cross blocks and the zero fantasy block (their Sigma entries are no longer needed)
    const double hs = 0.5 * gs;
    for (int idx = tid; idx < qt * qt; idx += KG_THREADS) {
        const int i = idx / qt, j = idx - i * qt;
        if (i < q && j < q) continue;
        double v = 0.0;
        if (i < q) v = hs * sV[(j - q) * ld + i];
        else if (j < q) v = hs * sV[(i - q) * ld + j];
        blk[idx] = v;
    }
    // L_bar, lower triangle over the leading block, fantasies in order
    for (int idx = tid; idx < q * q; idx += KG_THREADS) {
        const int i = idx / q, j = idx - i * q;
        if (j > i) continue;
        double s = 0.0;
        for (int f = 0; f < nf; f++) s = fma(sV[f * ld + i], sW[f * ld + j], s);
        blk[(size_t)i * qt + j] = -gs * s;
    }
    __syncthreads();
    block_chol_adjoint<KG_THREADS>(blk, q, qt, sL, lq);
}

inline cudaError_t launch_kg_block(const KgArgs& a, cudaStream_t st) {
    if (a.nb <= 0) return cudaSuccess;
    count_launch();
    const size_t smem = kg_smem_bytes(a.q, a.nf);
    cudaError_t e = cudaFuncSetAttribute(kg_block_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    kg_block_kernel<<<(unsigned)a.nb, KG_THREADS, smem, st>>>(a);
    return cudaGetLastError();
}

}  // namespace gpp
