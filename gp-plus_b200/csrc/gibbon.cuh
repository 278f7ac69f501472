// K4g: GIBBON, the lower bound of max-value entropy search (gpp_gibbon_qbatch; botorch's
// qLowerBoundMaxValueEntropy and, with target rows, qMultiFidelityLowerBoundMaxValueEntropy; Moss et al., 2021), and the
// max-value quartiles behind botorch's _sample_max_value_Gumbel (gpp_max_value_quartiles).
//
// Each t-batch t holds q_tot rows: the q actual points x_1..x_q, then (projected) their copies g_1..g_q at the target
// fidelity; tau(i) = q + i when projected, i otherwise.  One CTA per t-batch, after qbatch_syrk_kernel has written the
// latent q_tot x q_tot block Sigma (no noise).  With eps = 1e-8, sigma = +1 / -1 to maximise / minimise and the K
// max-value samples m_k (samples of max sigma f, shared by every t-batch):
//   V = Sigma[0:q, 0:q] + diag(n_i)             n_i the noise of row i's group, added here in place
//   L L^T = V + j_t I                            j_t the first rung of 0, 1e-8, 1e-7, 1e-6 that factors
//   v_i = max(V_ii, eps)   s_i^2 = max(Sigma_tau tau, eps)   c_i = Sigma_i tau   rho_i^2 = c_i^2 / (v_i s_i^2)
//   gamma_ik = (m_k - sigma mu_tau) / s_i        r_ik = phi(gamma_ik) / max(Phi(gamma_ik), eps)
//   Q_i = -(1/2K) sum_k log max(1 - rho_i^2 r_ik (gamma_ik + r_ik), eps)      quality: 1/2 log(v_i / Var(y_i | g <= m))
//   D   = sum_i (log L_ii - 1/2 log (V + j_t I)_ii)                            1/2 log det of the correlation matrix
//   v_t = D + sum_i Q_i
// The noiseless diagonal is saved before the noise is added, since s_i^2 and c_i read it when tau(i) = i.
// For the gradient, the two inputs of the q-batch backward (a clamped factor has zero derivative):
//   L_bar = diag(1 / L_ii) through block_chol_adjoint, then -1/2 / (V + j_t I)_ii on the diagonal: D's Sigma_bar
//   Q_i's adjoints of v_i, s_i^2 and c_i on Sigma_ii, Sigma_tau tau and (split evenly over both triangles)
//   Sigma_i tau; mu_bar[tau(i)] from gamma; every other entry 0
// Sigma_bar overwrites Sigma and mu_bar goes to the chunk's mean-gradient rows.
//
// Warp w owns rows i = w, w + 8, ...; its lanes take the samples k = lane, lane + 32, ... in order and combine their
// sums by a fixed butterfly, and every other sum runs in an order fixed by the t-batch's own indices, so a t-batch's
// outputs do not depend on the other t-batches of the call or on the chunk split.
#pragma once
#include "qbatch.cuh"

namespace gpp {

constexpr int GB_THREADS = 256;
constexpr double GB_EPS = 1e-8;  // botorch's CLAMP_LB

// doubles of dynamic shared memory: L [q x (q+1)], the noiseless diagonal [q_tot], then per actual row V_ii, Q_i and
// the adjoints of mu_tau, s^2, v and c
inline size_t gibbon_smem_bytes(int q, int q_tot) {
    return sizeof(double) * ((size_t)q * (q + 1) + q_tot + 6 * (size_t)q);
}

struct GibbonArgs {
    double* blk;           // [nb][q_tot][q_tot]: latent Sigma_t in; Sigma_bar_t out when grad
    const double* mu;      // chunk means in the tile layout (predict_finish_kernel)
    double* gm;            // chunk mean gradients in the tile layout (grad)
    const int* noise_idx;  // chunk noise groups in the tile layout, or NULL (group 0)
    const double* noise;
    int n_noise;
    const double* mv;      // [K] max-value samples
    int K;
    int q, q_tot, qpt;     // actual rows, rows per t-batch, t-batches per 128-row tile
    long long nb;          // t-batches in the chunk
    double sgn;            // +1 maximise, -1 minimise
    int grad;
    double* value;         // [nb]
    double* jitter;        // [nb]
    int* info;             // |= 1: a t-batch is not positive definite after the ladder, |= 2: NaN
};

__global__ void __launch_bounds__(GB_THREADS) gibbon_block_kernel(const GibbonArgs a) {
    extern __shared__ double gb_sm[];
    __shared__ int s_fail;
    const int q = a.q, qt = a.q_tot, tid = threadIdx.x, lq = q + 1, proj = qt != q;
    const int lane = tid & 31, warp = tid >> 5;
    double* sL = gb_sm;         // [q][q+1]
    double* sD = sL + q * lq;   // [q_tot] noiseless diagonal of Sigma
    double* sV = sD + qt;       // [q] V_ii
    double* sQ = sV + q;        // [q] Q_i
    double* sMb = sQ + q;       // [q] mu_bar of row tau(i)
    double* sSb = sMb + q;      // [q] adjoint of Sigma_tau tau
    double* sVb = sSb + q;      // [q] adjoint of V_ii
    double* sCb = sVb + q;      // [q] adjoint of c_i
    const long long t = blockIdx.x;
    const long long r0 = (t / a.qpt) * CT + (t % a.qpt) * qt;  // first row of t in the tile layout
    double* blk = a.blk + t * qt * qt;

    for (int i = tid; i < qt; i += GB_THREADS) {
        if (isnan(a.mu[r0 + i])) atomicOr(a.info, 2);
        sD[i] = blk[(size_t)i * qt + i];
    }
    __syncthreads();
    for (int i = tid; i < q; i += GB_THREADS) {
        const int gr = a.noise_idx ? a.noise_idx[r0 + i] : 0;
        const double v = sD[i] + ((gr >= 0 && gr < a.n_noise) ? a.noise[gr] : 0.0);
        blk[(size_t)i * qt + i] = v;
        sV[i] = v;
    }
    const double jit = block_ladder_chol<GB_THREADS>(blk, q, qt, sL, lq, &s_fail);
    if (s_fail) {
        if (tid == 0) {
            atomicOr(a.info, s_fail);
            a.value[t] = 0.0;
            a.jitter[t] = jit;
        }
        return;  // uniform across the CTA
    }
    const double inv2k = 0.5 / (double)a.K;
    for (int i = warp; i < q; i += GB_THREADS / 32) {
        const int tau = proj ? q + i : i;
        const double vraw = sV[i], s2raw = sD[tau];
        const double v = fmax(vraw, GB_EPS), s2 = fmax(s2raw, GB_EPS), s = sqrt(s2);
        const double c = proj ? blk[(size_t)i * qt + tau] : sD[i];
        const double rho2 = c * c / (v * s2);
        const double smu = a.sgn * a.mu[r0 + tau];
        double sl = 0.0, sh = 0.0, sg = 0.0, sgg = 0.0;
        for (int k = lane; k < a.K; k += 32) {
            const double g = (a.mv[k] - smu) / s;
            const double cdf = normcdf(g);
            const bool cl = !(cdf > GB_EPS);
            const double r = exp(-0.5 * g * g) * 0.3989422804014327 / (cl ? GB_EPS : cdf);
            const double hh = r * (g + r);
            const double am = 1.0 - rho2 * hh;
            if (am > GB_EPS) {
                sl += log(am);
                const double rp = cl ? -g * r : -hh;  // dr/dgamma
                const double hp = fma(rp, g + 2.0 * r, r);  // dh/dgamma
                sh += hh / am;
                sg += hp / am;
                sgg = fma(g, hp / am, sgg);
            } else {
                sl += log(GB_EPS);
            }
        }
        for (int o = 16; o > 0; o >>= 1) {
            sl += __shfl_xor_sync(0xffffffffu, sl, o);
            sh += __shfl_xor_sync(0xffffffffu, sh, o);
            sg += __shfl_xor_sync(0xffffffffu, sg, o);
            sgg += __shfl_xor_sync(0xffffffffu, sgg, o);
        }
        if (lane == 0) {
            sQ[i] = -inv2k * sl;
            const double grho = inv2k * sh;            // dQ / d rho^2
            const double ggam = inv2k * rho2 * sg;     // sum_k dQ / d gamma_k
            const double ggg = inv2k * rho2 * sgg;     // sum_k gamma_k dQ / d gamma_k
            sMb[i] = -a.sgn * ggam / s;
            sSb[i] = s2raw > GB_EPS ? -grho * rho2 / s2 - 0.5 * ggg / s2 : 0.0;
            sVb[i] = vraw > GB_EPS ? -grho * rho2 / v : 0.0;
            sCb[i] = grho * 2.0 * c / (v * s2);
        }
    }
    __syncthreads();
    if (tid == 0) {
        double d = 0.0;
        for (int i = 0; i < q; i++) d += log(sL[i * lq + i]) - 0.5 * log(sV[i] + jit);
        for (int i = 0; i < q; i++) d += sQ[i];
        if (isnan(d)) atomicOr(a.info, 2);
        a.value[t] = d;
        a.jitter[t] = jit;
    }
    if (!a.grad) return;
    for (int j = tid; j < qt; j += GB_THREADS) a.gm[r0 + j] = proj ? (j < q ? 0.0 : sMb[j - q]) : sMb[j];
    // L_bar = diag(1 / L_ii) over the leading block, 0 everywhere else
    for (int idx = tid; idx < qt * qt; idx += GB_THREADS) {
        const int i = idx / qt, j = idx - i * qt;
        blk[idx] = (i == j && i < q) ? 1.0 / sL[i * lq + i] : 0.0;
    }
    __syncthreads();
    block_chol_adjoint<GB_THREADS>(blk, q, qt, sL, lq);
    __syncthreads();
    for (int i = tid; i < q; i += GB_THREADS) {
        double* di = blk + (size_t)i * qt + i;
        *di += sVb[i] - 0.5 / (sV[i] + jit);
        if (proj) {
            const int tau = q + i;
            blk[(size_t)tau * qt + tau] = sSb[i];
            blk[(size_t)i * qt + tau] = 0.5 * sCb[i];
            blk[(size_t)tau * qt + i] = 0.5 * sCb[i];
        } else {
            *di += sSb[i] + sCb[i];
        }
    }
}

inline cudaError_t launch_gibbon_block(const GibbonArgs& a, cudaStream_t st) {
    if (a.nb <= 0) return cudaSuccess;
    count_launch();
    const size_t smem = gibbon_smem_bytes(a.q, a.q_tot);
    cudaError_t e = cudaFuncSetAttribute(gibbon_block_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    gibbon_block_kernel<<<(unsigned)a.nb, GB_THREADS, smem, st>>>(a);
    return cudaGetLastError();
}

// ---- max-value quartiles: l(y) = sum_j log Phi((y - sigma mu_j) / s_j) = log p for p = 1/4, 1/2, 3/4 ----
//
// mv_range_kernel: per block, min sigma mu_j, max sigma mu_j, max s_j and a flag for a non-finite marginal (exact in
// any order); mv_loglik_kernel: per block, l at the first npts of the MV_PTS points (1 while the bracket widens, since
// only l(hi) is asked, 3 while it is bisected), each thread's terms in increasing j and the block's by a fixed tree;
// mv_step_kernel (one block) sums the block partials in block order and moves the brackets.  The grid of both
// per-block kernels depends only on m, so the quartiles do not depend on how the marginals were computed in chunks.

constexpr int MV_THREADS = 256;
constexpr int MV_PTS = 3;

inline int mv_blocks(long long m) { return (int)std::min<long long>((m + MV_THREADS - 1) / MV_THREADS, 592); }

// log Phi(z), accurate in the lower tail through erfcx
__device__ __forceinline__ double log_ndtr(double z) {
    if (z < 0.0) {
        const double u = -z * 0.7071067811865476;
        return log(0.5 * erfcx(u)) - u * u;
    }
    return log1p(-0.5 * erfc(z * 0.7071067811865476));
}

// state: [0] lo, [1] hi, [2..4] the quartile brackets' lower ends, [5..7] their upper ends, [8..10] the points at
// which l is evaluated next, [11] the widening flag
constexpr int MV_STATE = 12;

__global__ void __launch_bounds__(MV_THREADS) mv_range_kernel(const double* mu, const double* var, long long m,
                                                              double sgn, double* part) {
    __shared__ double s_lo[MV_THREADS], s_hi[MV_THREADS], s_sd[MV_THREADS], s_nan[MV_THREADS];
    const int tid = threadIdx.x;
    double lo = INFINITY, hi = -INFINITY, sd = 0.0, nan = 0.0;
    for (long long j = (long long)blockIdx.x * MV_THREADS + tid; j < m; j += (long long)gridDim.x * MV_THREADS) {
        const double u = sgn * mu[j], s = sqrt(var[j]);
        if (!isfinite(u) || !isfinite(s)) nan = 1.0;
        lo = fmin(lo, u);
        hi = fmax(hi, u);
        sd = fmax(sd, s);
    }
    s_lo[tid] = lo;
    s_hi[tid] = hi;
    s_sd[tid] = sd;
    s_nan[tid] = nan;
    __syncthreads();
    for (int o = MV_THREADS / 2; o > 0; o >>= 1) {
        if (tid < o) {
            s_lo[tid] = fmin(s_lo[tid], s_lo[tid + o]);
            s_hi[tid] = fmax(s_hi[tid], s_hi[tid + o]);
            s_sd[tid] = fmax(s_sd[tid], s_sd[tid + o]);
            s_nan[tid] = fmax(s_nan[tid], s_nan[tid + o]);
        }
        __syncthreads();
    }
    if (tid == 0) {
        double* p = part + 4 * (size_t)blockIdx.x;
        p[0] = s_lo[0];
        p[1] = s_hi[0];
        p[2] = s_sd[0];
        p[3] = s_nan[0];
    }
}

// one block: the bracket lo = min sigma mu - 5 max s, hi = max sigma mu + 5 max s; *nan_out = 1 on a NaN or infinite
// marginal
__global__ void mv_range_finish_kernel(const double* part, int nblk, double* state, int* nan_out) {
    if (threadIdx.x != 0) return;
    double lo = INFINITY, hi = -INFINITY, sd = 0.0, nan = 0.0;
    for (int b = 0; b < nblk; b++) {
        lo = fmin(lo, part[4 * b]);
        hi = fmax(hi, part[4 * b + 1]);
        sd = fmax(sd, part[4 * b + 2]);
        nan = fmax(nan, part[4 * b + 3]);
    }
    *nan_out = nan > 0.0 ? 1 : 0;
    state[0] = lo - 5.0 * sd;
    state[1] = hi + 5.0 * sd;
    for (int p = 0; p < MV_PTS; p++) state[8 + p] = state[1];
}

__global__ void __launch_bounds__(MV_THREADS) mv_loglik_kernel(const double* mu, const double* var, long long m,
                                                               double sgn, const double* state, int npts,
                                                               double* part) {
    __shared__ double s_acc[MV_PTS][MV_THREADS];
    const int tid = threadIdx.x;
    double y[MV_PTS], acc[MV_PTS];
    for (int p = 0; p < MV_PTS; p++) {
        y[p] = state[8 + p];
        acc[p] = 0.0;
    }
    for (long long j = (long long)blockIdx.x * MV_THREADS + tid; j < m; j += (long long)gridDim.x * MV_THREADS) {
        const double u = sgn * mu[j], inv_s = 1.0 / sqrt(var[j]);
#pragma unroll
        for (int p = 0; p < MV_PTS; p++)  // a fixed trip count keeps y and acc in registers
            if (p < npts) acc[p] += log_ndtr((y[p] - u) * inv_s);
    }
    for (int p = 0; p < MV_PTS; p++) s_acc[p][tid] = acc[p];
    __syncthreads();
    for (int o = MV_THREADS / 2; o > 0; o >>= 1) {
        if (tid < o)
            for (int p = 0; p < MV_PTS; p++) s_acc[p][tid] += s_acc[p][tid + o];
        __syncthreads();
    }
    if (tid < MV_PTS) part[(size_t)blockIdx.x * MV_PTS + tid] = s_acc[tid][0];
}

// one block.  widen: point 0 is hi; when l(hi) < log 3/4, hi += hi - lo and the flag is set, else the three brackets
// start at [lo, hi] and the points move to its middle.  Otherwise one bisection step of each bracket.
__global__ void mv_step_kernel(const double* part, int nblk, double* state, int widen) {
    if (threadIdx.x != 0) return;
    const double logp[MV_PTS] = {-1.3862943611198906, -0.6931471805599453, -0.2876820724517809};
    double l[MV_PTS];
    for (int p = 0; p < MV_PTS; p++) {
        double s = 0.0;
        for (int b = 0; b < nblk; b++) s += part[(size_t)b * MV_PTS + p];
        l[p] = s;
    }
    if (widen) {
        const double lo = state[0], hi = state[1];
        if (l[0] < logp[MV_PTS - 1]) {
            state[1] = hi + (hi - lo);
            for (int p = 0; p < MV_PTS; p++) state[8 + p] = state[1];
            state[11] = 1.0;
            return;
        }
        state[11] = 0.0;
        for (int p = 0; p < MV_PTS; p++) {
            state[2 + p] = lo;
            state[5 + p] = hi;
            state[8 + p] = 0.5 * (lo + hi);
        }
        return;
    }
    for (int p = 0; p < MV_PTS; p++) {
        if (l[p] < logp[p]) state[2 + p] = state[8 + p];
        else state[5 + p] = state[8 + p];
        state[8 + p] = 0.5 * (state[2 + p] + state[5 + p]);
    }
}

}  // namespace gpp
