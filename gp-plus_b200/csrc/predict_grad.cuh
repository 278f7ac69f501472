// K4g: derivatives of the predictive mean and variance with respect to the candidates' quantitative inputs
// (GP_Plus.predict_with_grad, models/gp_plus.py:626-628: autograd through predict back to Xtest).
//
// With xs* = (xq* - centre) * sqrt(w), s_j = |xs* - xs_j|^2, zeta_j the latent factor averaged over the n_pass
// tables and k*_j = sf2 zeta_j f(s_j):
//   d k*_j / d xq*_d  = 2 sf2 zeta_j f'(s_j) sqrt(w_d) (xs*_d - xs_jd)
//   d mu / d xq*_d    =      sum_j d k*_j / d xq*_d  alpha_j
//   d var / d xq*_d   = -2 * sum_j d k*_j / d xq*_d  v_j,     v = K_y^-1 k*  (one row of V = K* L^-T L^-1)
// k** = sf2 does not depend on x*.  The engine forms V with two DMMA products (dgemm_dmma.cuh); the tile kernel below
// regenerates s, f' and zeta per (candidate, training point) pair from the point panels, so no M x N derivative matrix
// is ever stored, and writes one partial per column tile and dimension; the finish kernel reduces them in a fixed
// order (deterministic: no floating-point atomics) and applies 2 sf2 sqrt(w_d), the -2 and the clamp of the variance.
#pragma once
#include "cov.cuh"

namespace gpp {

constexpr int PG_THREADS = 256;  // 128 candidate rows x 2 column halves (the two lanes of a row are adjacent)
constexpr int PG_MAX_DQP = 36;   // pad_dq(GPP_MAX_DQ)

struct PredGradArgs {
    const double* xs_r;   // candidates [mcp*dqp] (prep_points_kernel layout, padded rows are 0)
    const double* zpt_r;  // [n_pass][mcp*ZP]
    long long zs_r;       // pass stride of zpt_r
    const double* xs_c;   // training points [np*dqp]
    const double* zpt_c;  // [n_pass][np*ZP]
    long long zs_c;
    const double* alpha;  // [np]
    const double* V;      // [mcp][ldv]: row i = (K_y^-1 k*_i)^T
    long long ldv;
    int n_r, n_c;         // valid candidates / training points
    int dq, dqp, dz, n_pass;
    double* part_m;       // [tiles_c*dq][ldp]: sum_j f' zeta alpha_j (xs_id - xs_jd) over column tile tj
    double* part_v;       // [tiles_c*dq][ldp]: sum_j f' zeta v_ij  (xs_id - xs_jd)
    long long ldp;
};

// grid (tiles_c, tiles_r).  Thread (row, half) walks the 64 columns of its half of the training tile with its row's
// inputs and its dq pairs of accumulators in registers (DQB: compile-time bound on dq); the two halves of a row are
// combined with one shuffle, the same sum in both lanes.
template <int KIND, bool HAS_Z, int DQB>
__global__ void __launch_bounds__(PG_THREADS) predict_grad_tile_kernel(const PredGradArgs a) {
    __shared__ double sxj[CT * PG_MAX_DQP];
    __shared__ double sal[CT];
    const int tid = threadIdx.x;
    const int tj = blockIdx.x, ti = blockIdx.y;
    const int dq = a.dq, dqp = a.dqp;
    for (int k = tid; k < CT * dqp; k += PG_THREADS) sxj[k] = a.xs_c[(long long)tj * CT * dqp + k];
    for (int k = tid; k < CT; k += PG_THREADS) sal[k] = a.alpha[(long long)tj * CT + k];
    __syncthreads();

    const int rl = tid >> 1, h = tid & 1;
    const int row = ti * CT + rl;
    const int c0 = h * (CT / 2);
    int ncol = a.n_c - (tj * CT + c0);
    ncol = ncol < 0 ? 0 : (ncol > CT / 2 ? CT / 2 : ncol);
    if (row >= a.n_r) ncol = 0;

    double xi[DQB], am[DQB], av[DQB];
#pragma unroll
    for (int d = 0; d < DQB; d++) {
        xi[d] = d < dq ? a.xs_r[(long long)row * dqp + d] : 0.0;
        am[d] = 0.0;
        av[d] = 0.0;
    }
    const double* vrow = a.V + (long long)row * a.ldv + (long long)tj * CT + c0;
    const double inv_pass = 1.0 / (double)a.n_pass;

#pragma unroll 1
    for (int jj = 0; jj < ncol; jj++) {
        const int c = c0 + jj;
        const double* xj = sxj + c * dqp;
        double s = 0.0;
#pragma unroll
        for (int d = 0; d < DQB; d++)
            if (d < dq) {
                const double df = xi[d] - xj[d];
                s = fma(df, df, s);
            }
        s = clamp_dist<KIND>(s);
        double f, fp;
        kq_eval_fast<KIND>(s, f, fp);
        double q = fp;
        if (HAS_Z) {
            double zeta = 0.0;
            for (int p = 0; p < a.n_pass; p++) {
                const double* zr = a.zpt_r + p * a.zs_r + (long long)row * ZP;
                const double* zc = a.zpt_c + p * a.zs_c + ((long long)tj * CT + c) * ZP;
                double sz = 0.0;
#pragma unroll
                for (int k = 0; k < ZP; k++)
                    if (k < a.dz) {
                        const double dd = zr[k] - zc[k];
                        sz = fma(dd, dd, sz);
                    }
                zeta += exp_nonpos_dev(-0.5 * sz);
            }
            if (a.n_pass > 1) zeta *= inv_pass;
            q *= zeta;
        }
        const double cm = q * sal[c], cv = q * vrow[jj];
#pragma unroll
        for (int d = 0; d < DQB; d++)
            if (d < dq) {
                const double df = xi[d] - xj[d];
                am[d] = fma(cm, df, am[d]);
                av[d] = fma(cv, df, av[d]);
            }
    }
#pragma unroll
    for (int d = 0; d < DQB; d++)
        if (d < dq) {
            am[d] += __shfl_xor_sync(0xffffffffu, am[d], 1);
            av[d] += __shfl_xor_sync(0xffffffffu, av[d], 1);
        }
    double* out = h == 0 ? a.part_m : a.part_v;
#pragma unroll
    for (int d = 0; d < DQB; d++)
        if (d < dq) out[((long long)tj * dq + d) * a.ldp + row] = h == 0 ? am[d] : av[d];
}

struct PredGradFinishArgs {
    const double* part_m;
    const double* part_v;
    long long ldp;
    const double* rowsq;      // [tiles_c][ldr] row sums of squares of U = K* L^-T (the variance, for its clamp)
    long long ldr;
    int tiles_c;
    int m, dq;
    const double* w;          // [dq]
    double sf2;
    const int* noise_idx;     // [m] or NULL
    const double* noise;
    int n_noise;
    int include_noise;
    double min_var;
    double* d_mean;           // [m*dq] chunk-local
    double* d_var;
};

__global__ void __launch_bounds__(256) predict_grad_finish_kernel(const PredGradFinishArgs a) {
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i >= a.m) return;
    // the variance exactly as predict_finish_kernel forms it; fmax(var, min_var) passes the gradient where
    // var >= min_var (torch's clamp_min) and blocks it elsewhere
    double q = 0.0;
    for (int t = 0; t < a.tiles_c; t++) q += a.rowsq[(long long)t * a.ldr + i];
    double var = a.sf2 - q;
    if (a.include_noise) {
        int g = a.noise_idx ? a.noise_idx[i] : 0;
        if (g >= 0 && g < a.n_noise) var += a.noise[g];
    }
    const bool pass = var >= a.min_var;
    for (int d = 0; d < a.dq; d++) {
        double sm = 0.0, sv = 0.0;
        for (int t = 0; t < a.tiles_c; t++) {
            sm += a.part_m[((long long)t * a.dq + d) * a.ldp + i];
            sv += a.part_v[((long long)t * a.dq + d) * a.ldp + i];
        }
        const double c = 2.0 * a.sf2 * sqrt(a.w[d]);
        a.d_mean[(long long)i * a.dq + d] = c * sm;
        a.d_var[(long long)i * a.dq + d] = pass ? -2.0 * c * sv : 0.0;
    }
}

template <bool HAS_Z, int DQB>
inline void launch_predict_grad_k(const PredGradArgs& a, int kind, dim3 grid, cudaStream_t st) {
    if (kind == KERNEL_EXPSQ) predict_grad_tile_kernel<KERNEL_EXPSQ, HAS_Z, DQB><<<grid, PG_THREADS, 0, st>>>(a);
    else if (kind == KERNEL_MATERN32) predict_grad_tile_kernel<KERNEL_MATERN32, HAS_Z, DQB><<<grid, PG_THREADS, 0, st>>>(a);
    else predict_grad_tile_kernel<KERNEL_MATERN52, HAS_Z, DQB><<<grid, PG_THREADS, 0, st>>>(a);
}

template <bool HAS_Z>
inline void launch_predict_grad_z(const PredGradArgs& a, int kind, dim3 grid, cudaStream_t st) {
    if (a.dq <= 8) launch_predict_grad_k<HAS_Z, 8>(a, kind, grid, st);
    else if (a.dq <= 16) launch_predict_grad_k<HAS_Z, 16>(a, kind, grid, st);
    else launch_predict_grad_k<HAS_Z, 32>(a, kind, grid, st);
}

inline cudaError_t launch_predict_grad(const PredGradArgs& a, int kind, int tiles_r, int tiles_c, cudaStream_t st) {
    if (tiles_r <= 0 || tiles_c <= 0 || a.dq <= 0) return cudaSuccess;
    if (a.dq > 32 || a.dqp > PG_MAX_DQP) return cudaErrorInvalidValue;
    count_launch();
    const dim3 grid(tiles_c, tiles_r);
    if (a.dz > 0) launch_predict_grad_z<true>(a, kind, grid, st);
    else launch_predict_grad_z<false>(a, kind, grid, st);
    return cudaGetLastError();
}

}  // namespace gpp
