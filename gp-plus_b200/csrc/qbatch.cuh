// K4q: joint posteriors of b independent t-batches of q candidates each and their input gradients
// (gpp_posterior_qbatch / gpp_posterior_qbatch_grad; botorch's posterior(X) on a [b, q, d] batch, which the reference
// GPR inherits from GPyTorchModel, models/gpregression.py:151-166).
//
// The engine lays the candidates out so that every 128-row tile of the prediction chunk holds qpt = 128 / q whole
// t-batches followed by padding rows, and runs the gpp_predict chunk loop on that layout with U = K* L^-T stored.
// Per t-batch t (rows of the tile, K** and K*_t regenerated from the point panels):
//   Sigma_t = K**_t - U_t U_t^T   (+ noise of each row on the diagonal when include_noise)
// and, for the vector-Jacobian product with upstream gradients g_mean and G_t (Gs_t = G_t + G_t^T, V = U L^-1):
//   d x_i = sum_n dk_in (g_mean_i alpha_n - W_in) + sum_{j != i in t} Gs_ij dk(x_i, x_j)/dx_i,   W = blockdiag(Gs) V
// with dk_in / dx_id = 2 sf2 zeta f'(s) sqrt(w_d) (xs_id - xs_nd) as in predict_grad.cuh.  Only the q x q diagonal
// blocks are ever formed: b q^2 Np flop for Sigma and for W, against b q Np^2 for U and V.
//
// Every value of a t-batch is computed from that t-batch's rows only and in an order fixed by its own row and column
// indices (sums over U columns from column 0, over t-batch members from member 0), never by its slot in the tile, so
// a t-batch's outputs do not depend on which other t-batches share the call or on the chunk split.
#pragma once
#include "cov.cuh"

namespace gpp {

constexpr int QB_THREADS = 256;      // 8 warps
constexpr int QB_KC = 32;            // U / V columns staged in shared memory per step
constexpr int QB_LDS = QB_KC + 4;    // row stride of the staged panel: DMMA fragment loads are bank-conflict free
constexpr int QB_MAXF = 17;          // lower 8x8 fragments of a 128-row tile (136) per warp, rounded up

// latent factor of the pair (i, j) averaged over the n_pass tables (1 without latent inputs)
__device__ __forceinline__ double qb_zeta(const double* zpt, long long zs, int dz, int n_pass, long long i,
                                          long long j) {
    if (dz <= 0) return 1.0;
    double zeta = 0.0;
    for (int p = 0; p < n_pass; p++) {
        const double* zi = zpt + p * zs + i * ZP;
        const double* zj = zpt + p * zs + j * ZP;
        double sz = 0.0;
#pragma unroll
        for (int k = 0; k < ZP; k++)
            if (k < dz) {
                const double dd = zi[k] - zj[k];
                sz = fma(dd, dd, sz);
            }
        zeta += exp_nonpos_dev(-0.5 * sz);
    }
    return n_pass > 1 ? zeta * (1.0 / (double)n_pass) : zeta;
}

struct QSyrkArgs {
    const double* U;       // [mcp][ldu] U = K* L^-T of the chunk
    long long ldu;
    int kcols;             // training points n: columns [0, n) of U (the rest faces K_y's identity padding)
    const double* rowsq;   // [tiles_c][ldr] row sums of squares of U (gpp_predict's variance)
    long long ldr;
    int tiles_c;
    const double* xs;      // [mcp*dqp] candidate panels (prep_points_kernel)
    const double* zpt;     // [n_pass][zs]
    long long zs;
    int dq, dqp, dz, n_pass;
    double sf2;
    const int* noise_idx;  // [mcp] or NULL
    const double* noise;
    int n_noise, include_noise;
    int q, qpt;            // rows per t-batch, t-batches per tile
    long long nb;          // t-batches in the chunk
    double* cov;           // [nb][q][q]
};

// One CTA per 128-row tile: the lower 8x8 fragments that meet a diagonal block, accumulated on DMMA over the U columns,
// then Sigma = K** - U U^T written to both triangles (exactly symmetric), the diagonal from the row sums.  GRAM: the
// blocks of U U^T itself, diagonal included (only U, ldu, kcols, q, qpt, nb and cov are read; KIND is unused).
template <int KIND, bool GRAM = false>
__global__ void __launch_bounds__(QB_THREADS) qbatch_syrk_kernel(const QSyrkArgs a) {
    __shared__ double sU[CT * QB_LDS];
    __shared__ unsigned char frag[136][2];
    __shared__ int nfrag;
    const int tile = blockIdx.x, tid = threadIdx.x;
    const int warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
    const int q = a.q;
    const long long left = a.nb - (long long)tile * a.qpt;
    const int rows = (int)(left < a.qpt ? left : a.qpt) * q;  // valid rows of this tile
    if (tid == 0) {
        int n = 0;
        for (int R = 0; R * 8 < rows; R++)
            for (int C = 0; C <= R; C++)
                if ((R * 8) / q <= min(C * 8 + 7, rows - 1) / q) {
                    frag[n][0] = (unsigned char)R;
                    frag[n][1] = (unsigned char)C;
                    n++;
                }
        nfrag = n;
    }
    double acc[QB_MAXF][2];
#pragma unroll
    for (int s = 0; s < QB_MAXF; s++) acc[s][0] = acc[s][1] = 0.0;
    const double* Ut = a.U + (long long)tile * CT * a.ldu;
    for (int k0 = 0; k0 < a.kcols; k0 += QB_KC) {
        __syncthreads();
        for (int idx = tid; idx < CT * QB_KC; idx += QB_THREADS) {
            const int r = idx / QB_KC, c = idx % QB_KC;
            sU[r * QB_LDS + c] = (r < rows && k0 + c < a.kcols) ? Ut[(long long)r * a.ldu + k0 + c] : 0.0;
        }
        __syncthreads();
        const int nf = nfrag;
#pragma unroll
        for (int kk = 0; kk < QB_KC; kk += 4) {
#pragma unroll
            for (int s = 0; s < QB_MAXF; s++) {
                const int f = warp + 8 * s;
                if (f < nf) {
                    const int R = frag[f][0], C = frag[f][1];
                    dmma884(acc[s][0], acc[s][1], sU[(R * 8 + g) * QB_LDS + kk + t], sU[(C * 8 + g) * QB_LDS + kk + t]);
                }
            }
        }
    }
    __syncthreads();
    const int nf = nfrag;
#pragma unroll
    for (int s = 0; s < QB_MAXF; s++) {
        const int f = warp + 8 * s;
        if (f >= nf) continue;
        const int i = frag[f][0] * 8 + g;
#pragma unroll
        for (int e = 0; e < 2; e++) {
            const int j = frag[f][1] * 8 + 2 * t + e;
            if (i >= rows || j > i || i / q != j / q) continue;
            const int bt = i / q, li = i - bt * q, lj = j - bt * q;
            const long long gi = (long long)tile * CT + i, gj = (long long)tile * CT + j;
            double v;
            if (GRAM) {
                v = acc[s][e];
            } else if (i == j) {  // predict_finish_kernel's unclamped variance, bit for bit
                double qs = 0.0;
                for (int tc = 0; tc < a.tiles_c; tc++) qs += a.rowsq[(long long)tc * a.ldr + gi];
                v = a.sf2 - qs;
                if (a.include_noise) {
                    const int gr = a.noise_idx ? a.noise_idx[gi] : 0;
                    if (gr >= 0 && gr < a.n_noise) v += a.noise[gr];
                }
            } else {
                double sd = 0.0;
                for (int d = 0; d < a.dq; d++) {
                    const double df = a.xs[gi * a.dqp + d] - a.xs[gj * a.dqp + d];
                    sd = fma(df, df, sd);
                }
                double fv, fp;
                kq_eval_fast<KIND>(clamp_dist<KIND>(sd), fv, fp);
                v = a.sf2 * fv * qb_zeta(a.zpt, a.zs, a.dz, a.n_pass, gi, gj) - acc[s][e];
            }
            double* out = a.cov + ((long long)tile * a.qpt + bt) * q * q;
            out[li * q + lj] = v;
            out[lj * q + li] = v;
        }
    }
}

struct QWArgs {
    const double* V;  // [mcp][ldv] V = K* K_y^-1 of the chunk
    long long ldv;
    const double* G;  // [nb][q][q] upstream gradient of the covariance blocks
    int q, qpt;
    long long nb;
    double* W;        // [mcp][ldw] blockdiag(G + G^T) V; padding rows 0
    long long ldw;
};

// grid (Np / 32, tiles).  Warp w owns rows 16 w .. 16 w + 15 and the CTA's 32 columns.  The K loop of an 8-row fragment
// runs once per t-batch it meets, over that t-batch's members from member 0, so the sum behind every W entry has the
// same terms in the same DMMA k-slots wherever the t-batch sits in the tile (rows of other t-batches add exact zeros).
__global__ void __launch_bounds__(QB_THREADS) qbatch_w_kernel(const QWArgs a) {
    __shared__ double sV[CT * QB_LDS];
    const int tile = blockIdx.y, c0 = blockIdx.x * QB_KC, tid = threadIdx.x;
    const int warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
    const int q = a.q;
    const long long left = a.nb - (long long)tile * a.qpt;
    const int rows = (int)(left < a.qpt ? left : a.qpt) * q;
    const double* Vt = a.V + (long long)tile * CT * a.ldv + c0;
    for (int idx = tid; idx < CT * QB_KC; idx += QB_THREADS) {
        const int r = idx / QB_KC, c = idx % QB_KC;
        sV[r * QB_LDS + c] = r < rows ? Vt[(long long)r * a.ldv + c] : 0.0;
    }
    __syncthreads();
    for (int rr = 0; rr < 2; rr++) {
        const int r0 = (warp * 2 + rr) * 8;
        const int i = r0 + g;
        double acc[4][2];
#pragma unroll
        for (int c = 0; c < 4; c++) acc[c][0] = acc[c][1] = 0.0;
        if (r0 < rows) {
            const int bi = i < rows ? i / q : -1;
            const int b_hi = min(r0 + 7, rows - 1) / q;
            for (int bt = r0 / q; bt <= b_hi; bt++) {
                const double* Gb = a.G + ((long long)tile * a.qpt + bt) * q * q;
                const int k0 = bt * q, li = i - k0;
                for (int kl = 0; kl < q; kl += 4) {
                    const int lk = kl + t;
                    const bool in = lk < q;
                    const double af = (bi == bt && in) ? Gb[li * q + lk] + Gb[lk * q + li] : 0.0;
#pragma unroll
                    for (int c = 0; c < 4; c++) {
                        const double bf = in ? sV[(k0 + lk) * QB_LDS + c * 8 + g] : 0.0;
                        dmma884(acc[c][0], acc[c][1], af, bf);
                    }
                }
            }
        }
        double* wr = a.W + ((long long)tile * CT + i) * a.ldw + c0 + 2 * t;
#pragma unroll
        for (int c = 0; c < 4; c++) {
            double2 v;
            v.x = acc[c][0];
            v.y = acc[c][1];
            *reinterpret_cast<double2*>(wr + c * 8) = v;
        }
    }
}

struct QInArgs {
    const double* xs;  // [mcp*dqp]
    const double* zpt;
    long long zs;
    int dq, dqp, dz, n_pass;
    const double* G;   // [nb][q][q]
    int q, qpt;
    long long nb;
    int rows;          // mcp
    double* part_k;    // [mcp][dq]: sum_{j != i in t} Gs_ij f'(s_ij) zeta_ij (xs_id - xs_jd)
};

// K** term of the gradient: one warp per candidate row, lane d holds input dimension d (dq <= 32); s_ij is reduced
// with a butterfly, which leaves the same value in every lane.
template <int KIND>
__global__ void __launch_bounds__(256) qbatch_inbatch_grad_kernel(const QInArgs a) {
    const long long i = ((long long)blockIdx.x * 256 + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (i >= a.rows) return;
    const int q = a.q, r = (int)(i % CT), slot = r / q;
    const long long bt = (i / CT) * a.qpt + slot;
    const bool own = lane < a.dq;
    double acc = 0.0;
    if (slot < a.qpt && bt < a.nb) {
        const int li = r - slot * q;
        const long long j0 = i - li;
        const double* Gb = a.G + bt * q * q;
        const double xi = own ? a.xs[i * a.dqp + lane] : 0.0;
        for (int lj = 0; lj < q; lj++) {
            if (lj == li) continue;
            const long long j = j0 + lj;
            const double df = own ? xi - a.xs[j * a.dqp + lane] : 0.0;
            double s = df * df;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
            double fv, fp;
            kq_eval_fast<KIND>(clamp_dist<KIND>(s), fv, fp);
            const double cf = (Gb[li * q + lj] + Gb[lj * q + li]) * fp * qb_zeta(a.zpt, a.zs, a.dz, a.n_pass, i, j);
            acc = fma(cf, df, acc);
        }
    }
    if (own) a.part_k[i * a.dq + lane] = acc;
}

struct QFinishArgs {
    const double* part_m;  // [tiles_c*dq][ldp] from predict_grad_tile_kernel (alpha)
    const double* part_v;  // [tiles_c*dq][ldp] from predict_grad_tile_kernel (W)
    long long ldp;
    int tiles_c;
    const double* part_k;  // [m][dq]
    const double* g_mean;  // [m] or NULL
    int m, dq;
    const double* w;       // [dq]
    double sf2;
    double* d_x;           // [m][dq]
};

// d x_id = 2 sf2 sqrt(w_d) (g_mean_i sum_t part_m - sum_t part_v + part_k), column tiles summed in order
__global__ void __launch_bounds__(256) qbatch_grad_finish_kernel(const QFinishArgs a) {
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i >= a.m) return;
    const double gm = a.g_mean ? a.g_mean[i] : 0.0;
    for (int d = 0; d < a.dq; d++) {
        double sm = 0.0, sv = 0.0;
        for (int t = 0; t < a.tiles_c; t++) {
            sm += a.part_m[((long long)t * a.dq + d) * a.ldp + i];
            sv += a.part_v[((long long)t * a.dq + d) * a.ldp + i];
        }
        const double c = 2.0 * a.sf2 * sqrt(a.w[d]);
        a.d_x[(long long)i * a.dq + d] = c * ((gm * sm - sv) + a.part_k[(long long)i * a.dq + d]);
    }
}

inline cudaError_t launch_qbatch_syrk(const QSyrkArgs& a, int kind, int tiles, cudaStream_t st) {
    count_launch();
    if (kind == KERNEL_EXPSQ) qbatch_syrk_kernel<KERNEL_EXPSQ><<<tiles, QB_THREADS, 0, st>>>(a);
    else if (kind == KERNEL_MATERN32) qbatch_syrk_kernel<KERNEL_MATERN32><<<tiles, QB_THREADS, 0, st>>>(a);
    else qbatch_syrk_kernel<KERNEL_MATERN52><<<tiles, QB_THREADS, 0, st>>>(a);
    return cudaGetLastError();
}

// the q x q diagonal blocks of U U^T over columns [0, kcols) (gpp_nipv_qbatch's C_t^T C_t)
inline cudaError_t launch_qbatch_gram(const QSyrkArgs& a, int tiles, cudaStream_t st) {
    count_launch();
    qbatch_syrk_kernel<KERNEL_EXPSQ, true><<<tiles, QB_THREADS, 0, st>>>(a);
    return cudaGetLastError();
}

inline cudaError_t launch_qbatch_inbatch_grad(const QInArgs& a, int kind, cudaStream_t st) {
    count_launch();
    const int blocks = (int)(((long long)a.rows * 32 + 255) / 256);
    if (kind == KERNEL_EXPSQ) qbatch_inbatch_grad_kernel<KERNEL_EXPSQ><<<blocks, 256, 0, st>>>(a);
    else if (kind == KERNEL_MATERN32) qbatch_inbatch_grad_kernel<KERNEL_MATERN32><<<blocks, 256, 0, st>>>(a);
    else qbatch_inbatch_grad_kernel<KERNEL_MATERN52><<<blocks, 256, 0, st>>>(a);
    return cudaGetLastError();
}

// ---- per-t-batch block factor and its adjoint, for kernels that run one CTA of NT threads per t-batch ----

// L = chol(A + j I) of the leading n x n block of A (row-major, leading dimension lda, lower triangle read) into sL
// [n][lq] in shared memory, j the first rung of 0, 1e-8, 1e-7, 1e-6 whose pivots are all > 0 (dpotrf's test, the
// psd_safe_cholesky ladder); each rung restarts from A.  Called by every thread of the CTA; returns j with *s_fail
// (shared) 0 when that rung factored, 1 when every rung failed and 2 on a NaN pivot, the same for all threads.
template <int NT>
__device__ __forceinline__ double block_ladder_chol(const double* A, int n, int lda, double* sL, int lq, int* s_fail) {
    const int tid = threadIdx.x;
    double jit = 0.0;
    for (int rung = 0;; rung++) {
        jit = rung == 0 ? 0.0 : (rung == 1 ? 1e-8 : (rung == 2 ? 1e-7 : 1e-6));
        __syncthreads();
        for (int idx = tid; idx < n * n; idx += NT) {
            const int i = idx / n, j = idx - i * n;
            if (j <= i) sL[i * lq + j] = A[i * lda + j] + (i == j ? jit : 0.0);
        }
        if (tid == 0) *s_fail = 0;
        __syncthreads();
        for (int k = 0; k < n; k++) {
            if (tid == 0) {
                const double d = sL[k * lq + k];
                if (isnan(d)) *s_fail = 2;
                else if (!(d > 0.0)) *s_fail = 1;
                else sL[k * lq + k] = sqrt(d);
            }
            __syncthreads();
            if (*s_fail) break;
            const double lkk = sL[k * lq + k];
            for (int i = k + 1 + tid; i < n; i += NT) sL[i * lq + k] /= lkk;
            __syncthreads();
            const int m = n - k - 1;
            for (int idx = tid; idx < m * m; idx += NT) {
                const int i = k + 1 + idx / m, j = k + 1 + idx % m;
                if (j <= i) sL[i * lq + j] = fma(-sL[i * lq + k], sL[j * lq + k], sL[i * lq + j]);
            }
            __syncthreads();
        }
        if (!*s_fail || *s_fail == 2 || rung == 3) return jit;
    }
}

// torch's cholesky backward on the leading n x n block of B (leading dimension ldb), in place: L_bar in its lower
// triangle in, A_bar = L^-T Phi(L^T L_bar) L^-1 out, exactly symmetric (Phi keeps the lower triangle and halves its
// diagonal, then mirrors it).  L is block_ladder_chol's factor; n <= NT; called by every thread after a barrier that
// follows the last write of L_bar.
template <int NT>
__device__ __forceinline__ void block_chol_adjoint(double* B, int n, int ldb, const double* sL, int lq) {
    const int tid = threadIdx.x;
    // M = tril(L^T L_bar), row i from rows k >= i of L_bar, in place in increasing i
    for (int i = 0; i < n; i++) {
        double mv = 0.0;
        if (tid <= i)
            for (int k = i; k < n; k++) mv = fma(sL[k * lq + i], B[k * ldb + tid], mv);
        __syncthreads();
        if (tid <= i) B[i * ldb + tid] = mv;
    }
    __syncthreads();
    // P = Phi(M) mirrored: P_ij = P_ji = M_ij / 2 (j <= i)
    for (int idx = tid; idx < n * n; idx += NT) {
        const int i = idx / n, j = idx - i * n;
        if (j <= i) {
            const double v = 0.5 * B[i * ldb + j];
            B[i * ldb + j] = v;
            B[j * ldb + i] = v;
        }
    }
    __syncthreads();
    // Z = P L^-1 row by row (Z L = P), in place
    if (tid < n) {
        double* zr = B + tid * ldb;
        for (int j = n - 1; j >= 0; j--) {
            double v = zr[j];
            for (int k = j + 1; k < n; k++) v = fma(-zr[k], sL[k * lq + j], v);
            zr[j] = v / sL[j * lq + j];
        }
    }
    __syncthreads();
    // G = L^-T Z column by column (L^T G = Z), in place
    if (tid < n) {
        for (int j = n - 1; j >= 0; j--) {
            double v = B[j * ldb + tid];
            for (int k = j + 1; k < n; k++) v = fma(-sL[k * lq + j], B[k * ldb + tid], v);
            B[j * ldb + tid] = v / sL[j * lq + j];
        }
    }
    __syncthreads();
    for (int idx = tid; idx < n * n; idx += NT) {  // exact symmetry
        const int i = idx / n, j = idx - i * n;
        if (j < i) {
            const double v = 0.5 * (B[i * ldb + j] + B[j * ldb + i]);
            B[i * ldb + j] = v;
            B[j * ldb + i] = v;
        }
    }
}

}  // namespace gpp
