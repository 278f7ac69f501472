// K4a: Monte-Carlo batch acquisition on the t-batch posteriors of qbatch.cuh (gpp_acq_qbatch; botorch's qEI, qNEI and
// qUCB with a sampler whose base samples E [S x q] are shared by every t-batch).
//
// One CTA per t-batch t, after qbatch_syrk_kernel has written Sigma_t into the chunk's block buffer:
//   L_t = chol(Sigma_t + j_t I)   j_t the first rung of 0, 1e-8, 1e-7, 1e-6 whose pivots are all > 0 (dpotrf's test)
//   y_s = mu_t + L_t e_s,  v_t = (1/S) sum_s u(y_s)   (u: qEI, qNEI or qUCB utility, sigma = +1 / -1 to max / min)
// and, for the gradient, the reverse of those steps: each u is one-hot in y (two-hot for qNEI), so
//   mu_bar = (1/S) sum_s g_s,  L_bar = (1/S) sum_s g_s e_s^T   (per-row accumulations of base-sample rows)
//   G_t = L^-T Phi(L^T L_bar) L^-1, symmetrised   (torch's cholesky backward: Phi keeps the lower triangle and halves
//                                                  its diagonal, then mirrors it)
// G_t overwrites Sigma_t and mu_bar goes to the chunk's mean-gradient rows: the inputs of the q-batch backward.
//
// Every sum runs in an order fixed by the t-batch's own row, column and sample indices, so a t-batch's value, jitter
// and gradient do not depend on the other t-batches of the call or on the chunk split.
#pragma once
#include "qbatch.cuh"

namespace gpp {

constexpr int QA_THREADS = 256;
constexpr int QA_ROWS = 2048;  // base-sample entries (rows x q) staged in shared memory per step
constexpr int QA_MAXS = 256;   // base-sample rows per step

__device__ __forceinline__ int qa_chunk(int q) { return max(1, min(QA_MAXS, QA_ROWS / q)); }

// doubles of dynamic shared memory: L [q x (q+1)], E and L E^T [SC x ld], mu and four per-sample arrays
inline size_t qa_smem_bytes(int q) {
    const int sc = std::max(1, std::min(QA_MAXS, QA_ROWS / q));
    const int ld = q | 1;
    return sizeof(double) * ((size_t)q * (q + 1) + 2 * (size_t)sc * ld + q + 3 * (size_t)sc) + sizeof(int) * 2 * sc;
}

struct QAcqArgs {
    double* blk;       // [nb][q][q]: Sigma_t in; G_t out when grad
    const double* mu;  // chunk means in the tile layout (predict_finish_kernel)
    double* gm;        // chunk mean gradients in the tile layout (grad)
    const double* E;   // [S][q] base samples
    long long S;
    int q, qpt, n_base;
    long long nb;      // t-batches in the chunk
    double sgn;        // +1 maximise, -1 minimise
    double best_f;     // qEI incumbent (scaled units)
    double cbeta;      // qUCB sqrt(beta pi / 2)
    int grad;
    double* value;     // [nb]
    double* jitter;    // [nb]
    int* info;         // |= 1: a t-batch is not positive definite after the ladder, |= 2: NaN
};

template <int KIND>
__global__ void __launch_bounds__(QA_THREADS) qacq_mc_kernel(const QAcqArgs a) {
    extern __shared__ double qa_sm[];
    __shared__ int s_fail;
    const int q = a.q, tid = threadIdx.x, sc = qa_chunk(q), ld = q | 1, lq = q + 1;
    double* sL = qa_sm;            // [q][q+1]
    double* sE = sL + q * lq;      // [sc][ld]
    double* sZ = sE + sc * ld;     // [sc][ld]  (L e_s)_i
    double* sMu = sZ + sc * ld;    // [q]
    double* sU = sMu + q;          // [sc] utility
    double* sWL = sU + sc;         // [sc] weight of the sample's row in L_bar
    double* sWM = sWL + sc;        // [sc] weight of the sample's row in mu_bar
    int* sI = (int*)(sWM + sc);    // [2 sc] row of the sample's utility (qNEI: baseline row second), -1 none
    const long long t = blockIdx.x;
    const long long r0 = (t / a.qpt) * CT + (t % a.qpt) * q;  // first row of t in the tile layout
    double* blk = a.blk + t * q * q;
    const int qc = q - a.n_base;   // candidate rows (qNEI: the rest are baseline rows)

    for (int i = tid; i < q; i += QA_THREADS) {
        sMu[i] = a.mu[r0 + i];
        if (isnan(sMu[i])) atomicOr(a.info, 2);
    }
    // L_t in shared memory (the ladder of block_ladder_chol)
    const double jit = block_ladder_chol<QA_THREADS>(blk, q, q, sL, lq, &s_fail);
    if (s_fail) {
        if (tid == 0) {
            atomicOr(a.info, s_fail);
            a.value[t] = 0.0;
            a.jitter[t] = jit;
        }
        return;  // uniform across the CTA
    }
    if (a.grad) {  // L_bar accumulates in the block (Sigma_t is no longer needed)
        __syncthreads();
        for (int idx = tid; idx < q * q; idx += QA_THREADS) blk[idx] = 0.0;
    }
    double vsum = 0.0, mbar = 0.0;  // vsum: lane 0 of warp 0; mbar: thread i < q owns mu_bar_i
    bool nan_seen = false;
    for (long long s0 = 0; s0 < a.S; s0 += sc) {
        const int ns = (int)min((long long)sc, a.S - s0);
        __syncthreads();
        for (int idx = tid; idx < ns * q; idx += QA_THREADS) {
            const int s = idx / q, c = idx - s * q;
            sE[s * ld + c] = a.E[(s0 + s) * q + c];
        }
        __syncthreads();
        for (int idx = tid; idx < ns * q; idx += QA_THREADS) {
            const int s = idx / q, i = idx - s * q;
            const double* Li = sL + i * lq;
            const double* e = sE + s * ld;
            double z = 0.0;
            for (int c = 0; c <= i; c++) z = fma(Li[c], e[c], z);
            sZ[s * ld + i] = z;
        }
        __syncthreads();
        for (int s = tid; s < ns; s += QA_THREADS) {
            const double* z = sZ + s * ld;
            double best = -INFINITY, u = 0.0, wl = 0.0, wm = 0.0;
            int bi = -1, bj = -1;
            if (KIND == GPP_QACQ_UCB) {
                for (int i = 0; i < q; i++) {
                    const double v = fma(a.cbeta, fabs(z[i]), a.sgn * sMu[i]);
                    nan_seen |= isnan(v);
                    if (v > best) best = v, bi = i;
                }
                u = best;
                if (bi >= 0) wl = z[bi] > 0.0 ? a.cbeta : (z[bi] < 0.0 ? -a.cbeta : 0.0), wm = a.sgn;
            } else {
                for (int i = 0; i < qc; i++) {
                    const double v = a.sgn * (sMu[i] + z[i]);
                    nan_seen |= isnan(v);
                    if (v > best) best = v, bi = i;
                }
                double ref = a.sgn * a.best_f;
                if (KIND == GPP_QACQ_NEI) {
                    ref = -INFINITY;
                    for (int j = qc; j < q; j++) {
                        const double v = a.sgn * (sMu[j] + z[j]);
                        nan_seen |= isnan(v);
                        if (v > ref) ref = v, bj = j;
                    }
                }
                u = best - ref;
                if (u > 0.0) wl = wm = a.sgn;
                else u = 0.0, bi = bj = -1;
            }
            sU[s] = u;
            sWL[s] = wl;
            sWM[s] = wm;
            sI[2 * s] = bi;
            sI[2 * s + 1] = bj;
        }
        __syncthreads();
        if (tid < 32) {  // the chunk's utilities: lane-strided partial sums, then a fixed butterfly
            double p = 0.0;
            for (int s = tid; s < ns; s += 32) p += sU[s];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) p += __shfl_xor_sync(0xffffffffu, p, o);
            vsum += p;
        }
        if (a.grad && tid < q) {  // column tid of L_bar and mu_bar_tid, samples in order
            const int c = tid;
            for (int s = 0; s < ns; s++) {
#pragma unroll
                for (int h = 0; h < 2; h++) {
                    const int r = sI[2 * s + h];
                    if (r < 0) continue;
                    const double sg = h ? -1.0 : 1.0;
                    if (c <= r) blk[r * q + c] = fma(sg * sWL[s], sE[s * ld + c], blk[r * q + c]);
                    if (c == r) mbar = fma(sg, sWM[s], mbar);
                }
            }
        }
    }
    if (nan_seen) atomicOr(a.info, 2);
    const double inv_s = 1.0 / (double)a.S;
    if (tid == 0) {
        a.value[t] = vsum * inv_s;
        a.jitter[t] = jit;
    }
    if (!a.grad) return;
    if (tid < q) {
        a.gm[r0 + tid] = mbar * inv_s;
        for (int r = tid; r < q; r++) blk[r * q + tid] *= inv_s;
    }
    __syncthreads();
    block_chol_adjoint<QA_THREADS>(blk, q, q, sL, lq);
}

template <int KIND>
inline cudaError_t launch_qacq_kind(const QAcqArgs& a, size_t smem, cudaStream_t st) {
    cudaError_t e = cudaFuncSetAttribute(qacq_mc_kernel<KIND>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    qacq_mc_kernel<KIND><<<(unsigned)a.nb, QA_THREADS, smem, st>>>(a);
    return cudaGetLastError();
}

inline cudaError_t launch_qacq(const QAcqArgs& a, int kind, cudaStream_t st) {
    if (a.nb <= 0) return cudaSuccess;
    count_launch();
    const size_t smem = qa_smem_bytes(a.q);
    if (kind == GPP_QACQ_EI) return launch_qacq_kind<GPP_QACQ_EI>(a, smem, st);
    if (kind == GPP_QACQ_NEI) return launch_qacq_kind<GPP_QACQ_NEI>(a, smem, st);
    return launch_qacq_kind<GPP_QACQ_UCB>(a, smem, st);
}

}  // namespace gpp
