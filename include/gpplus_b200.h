/*
 * gpplus_b200.h -- C ABI of the B200-native exact-GP engine behind GP+'s Python API.
 *
 * The reference (Bostanabad-Research-Group/GP-Plus) is pure Python and has no FFI of
 * its own: the seam is two Python call sites.  Every entry point below names the
 * reference call site it replaces (paths relative to the reference root).
 *
 *   - MLLObjective.fun            optim/mll_scipy.py:112-127   -> gpp_mll_grad
 *       (forward:  models/gp_plus.py:386-484, likelihood: likelihoods_noise/multifidelity.py:63-136,
 *        log_prob: optim/mll_scipy.py:37-39, backward: optim/mll_scipy.py:123)
 *   - GPR.predict                 models/gpregression.py:122-149 -> gpp_factorize + gpp_predict
 *   - GP_Plus.predict_with_grad   models/gp_plus.py:626-628      -> gpp_factorize + gpp_predict_grad
 *   - GPR.posterior (joint), MultivariateNormal.rsample
 *                                 models/gpregression.py:151-166 -> gpp_predict_joint, gpp_sample_posterior
 *   - GPR.posterior on [..., q, d] (botorch's posterior(X) for q-batch acquisition) and its backward
 *                                 models/gpregression.py:151-166 -> gpp_posterior_qbatch, gpp_posterior_qbatch_grad
 *   - botorch qEI / qNEI / qUCB (MC acquisition on posterior(X).rsample with shared base samples) and their
 *     gradients in X: GPR.acquisition_qbatch, bayesian_optimizations/qbatch.py -> gpp_acq_qbatch
 *   - botorch qNegIntegratedPosteriorVariance and its gradient in X: GPR.acquisition_qbatch(X, "qNIPV", mc_points)
 *                                 -> gpp_ipv_points, gpp_nipv_qbatch
 *   - botorch one-shot qKnowledgeGradient (cost-aware as qMultiFidelityKnowledgeGradient) and its gradient in X:
 *     GPR.knowledge_gradient, bayesian_optimizations/qbatch.py -> gpp_kg_qbatch
 *   - botorch qLowerBoundMaxValueEntropy / qMultiFidelityLowerBoundMaxValueEntropy (GIBBON) and its gradient in X, and
 *     the max-value samples of _sample_max_value_Gumbel: GPR.gibbon, GPR.sample_max_values,
 *     bayesian_optimizations/qbatch.py -> gpp_gibbon_qbatch, gpp_max_value_quartiles
 *   - AF_*_Engineering + argmax   bayesian_optimizations/AFs.py:102-159,
 *                                 bayesian_optimizations/BO_GP_plus.py:183-194 -> gpp_acq_argmax
 *   - covar_module(x).evaluate()  models/gp_plus.py:472-474      -> gpp_covariance
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer is a HOST pointer unless its name ends
 *     in _dev.  The library owns all device memory; callers keep ownership of host buffers.
 *   - all entry points return a status: GPP_OK, GPP_ERR_NOT_PD (Cholesky failed after the
 *     jitter ladder; Python raises NotPSDError), GPP_ERR_NAN (NaN in K; Python raises
 *     NanError), GPP_ERR_ARG, or GPP_ERR_CUDA (see gpp_last_error()).
 *     No exception crosses the boundary.  There is no CPU fallback.
 *   - a handle is bound to one device and one stream; handles are not thread-safe,
 *     distinct handles are (one handle per in-flight restart).
 *   - hyper-parameters are passed in their CONSTRAINED (natural) form; the raw->natural
 *     transforms and the log-priors are O(p) and stay on the host (Python).
 */
#ifndef GPPLUS_B200_H
#define GPPLUS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GPP_OK 0
#define GPP_ERR_NOT_PD 1
#define GPP_ERR_NAN 2
#define GPP_ERR_ARG 3
#define GPP_ERR_CUDA (-1)

/* quantitative-kernel family; s = sum_d w[d] * (x_id - x_jd)^2
 *   GPP_KERNEL_EXPSQ    k = exp(-s)                     (Rough_RBF: w = 10^omega, kernels/Rough_RBF.py:27-32;
 *                                                        RBFKernel: w = 0.5*exp(-2 raw), models/gp_plus.py:242-247)
 *   GPP_KERNEL_MATERN32 k = (1+sqrt3 r) exp(-sqrt3 r)   r = sqrt(s), w = 2*10^omega   (kernels/matern.py:4-5)
 *   GPP_KERNEL_MATERN52 k = (1+sqrt5 r+5/3 r^2) exp(-sqrt5 r)                         (kernels/matern.py:7-8)
 * the categorical part is always  exp(-0.5*||z_i - z_j||^2)  (fixed-lengthscale RBF on the
 * latent coordinates, models/gp_plus.py:219-226) and multiplies the quantitative kernel. */
#define GPP_KERNEL_EXPSQ 0
#define GPP_KERNEL_MATERN32 1
#define GPP_KERNEL_MATERN52 2

#define GPP_MAX_DQ 32   /* quantitative input columns */
#define GPP_MAX_DZ 4    /* latent (embedding) dimensions */

/* acquisition kinds, bayesian_optimizations/AFs.py */
#define GPP_ACQ_HF 0    /* sigma*u/cost                 AFs.py:135-159 */
#define GPP_ACQ_LF 1    /* sigma*pdf(u)/cost            AFs.py:102-132 */
#define GPP_ACQ_EI 2    /* sigma*(pdf(u)+u*cdf(u))/cost AFs.py:67-99   */

typedef struct gpp_handle gpp_handle;

/* Static description of one training set (GPR.__init__, models/gpregression.py:39-115;
 * index bookkeeping models/gp_plus.py:184-215). */
typedef struct gpp_problem {
    int64_t n;                /* training points */
    int32_t dq;               /* quantitative columns (<= GPP_MAX_DQ) */
    int32_t dz;               /* latent dimensions, 0 when there is no categorical input */
    int32_t n_combo;          /* rows of the latent table Z (level combinations), 0 if dz==0 */
    int32_t n_noise;          /* noise groups; 1 = homoskedastic GaussianLikelihood */
    int32_t n_mean;           /* mean constants; 0 = ZeroMean */
    int32_t kernel;           /* GPP_KERNEL_* */
    const double* xq;         /* [n*dq] row-major quantitative inputs */
    const double* y;          /* [n] targets, already min-max scaled (gpregression.py:67-69) */
    const int32_t* level_idx; /* [n] row of Z per point (perm_dict lookup, gp_plus.py:1085); NULL if dz==0 */
    const int32_t* noise_idx; /* [n] noise group per point (multifidelity.py:105-136); NULL = all 0 */
    const int32_t* mean_idx;  /* [n] mean constant per point, -1 = zero mean (gp_plus.py:529-534); NULL = all 0 */
    int32_t n_pass;           /* latent tables averaged into K: Sigma = (1/k) sum_p K(Z_p) -- the multi-pass ensemble
                               * covariance of the probabilistic embedding (gp_plus.py:387-399, 414-461, 474-482);
                               * 0 or 1 = one deterministic table */
} gpp_problem;

/* Hyper-parameters in natural form for one evaluation. */
typedef struct gpp_hyper {
    const double* w;        /* [dq]  distance weights (see GPP_KERNEL_*) */
    const double* z;        /* [n_pass*n_combo*dz] latent table(s) Z = zeta_table * A^T (gp_plus.py:436), NULL if dz==0 */
    double sigma_f2;        /* outputscale = softplus(raw) (gpregression.py:108-111) */
    const double* noise;    /* [n_noise] noise variances lb+exp(raw) (gpregression.py:59) */
    const double* beta;     /* [n_mean]  mean constants, NULL if n_mean==0 */
} gpp_hyper;

/* Result of one MLL(+gradient) evaluation.  nll is the DATA term only,
 *   nll = -log N(y; m, K + noise)   (optim/mll_scipy.py:38-39, not divided by n);
 * gradients are d nll / d(natural parameter); priors and chain rules to the raw
 * parameters are applied by the caller.  Gradient pointers may be NULL. */
typedef struct gpp_mll_result {
    double nll;
    double logdet;          /* log|K_y| */
    double quad;            /* (y-m)^T K_y^{-1} (y-m) */
    double jitter;          /* diagonal jitter that was needed (0, 1e-8, 1e-7 or 1e-6) */
    double d_sigma_f2;
    double* d_w;            /* [dq] */
    double* d_z;            /* [n_pass*n_combo*dz] */
    double* d_noise;        /* [n_noise] */
    double* d_beta;         /* [n_mean] */
} gpp_mll_result;

/* per-stage device times of the last gpp_mll_grad call, milliseconds (CUDA events) */
typedef struct gpp_timings {
    float covariance;       /* K1 fused covariance builder */
    float cholesky;         /* K2 blocked Cholesky incl. diagonal-block inverses */
    float trtri;            /* L^{-1} by recursive doubling */
    float solve;            /* alpha, quad, logdet */
    float lauum;            /* K^{-1} = L^{-T} L^{-1} */
    float gradient;         /* K3 fused gradient reduction */
    float total;
} gpp_timings;

/* per-handle counters since gpp_create (bench.py reports jitter-ladder retries separately, SURVEY 8d) */
typedef struct gpp_stats {
    int64_t evaluations;     /* gpp_mll_grad / gpp_objective / gpp_factorize calls */
    int64_t factorizations;  /* Cholesky attempts (evaluations + jitter retries) */
    int64_t jitter_retries;  /* attempts with jitter 1e-8 / 1e-7 / 1e-6 (psd_safe_cholesky ladder) */
    int64_t early_outs;      /* failed attempts abandoned right after the factorisation */
} gpp_stats;

int gpp_version(void);
int gpp_device_count(void);
const char* gpp_last_error(void);
/* number of CUDA kernels this library has launched in this process (bench.py's gpu_launches) */
long long gpp_launch_count(void);

/* gpp_destroy parks handles of small problems (<= 192 MB of device memory) in a per-process pool and gpp_create
 * hands a parked handle of the same shape and device back after re-uploading the training data: the multi-start
 * driver creates dozens of handles per fit and allocation / teardown would otherwise cost more than the fit.
 * gpp_pool_clear frees every parked handle (GPP_POOL=0 disables parking). */
int gpp_create(const gpp_problem* problem, int device, gpp_handle** out);
void gpp_destroy(gpp_handle* h);
void gpp_pool_clear(void);

/* replaces MLLObjective.fun (optim/mll_scipy.py:112-127) */
int gpp_mll_grad(gpp_handle* h, const gpp_hyper* hyper, int want_grad, gpp_mll_result* out);
int gpp_get_timings(gpp_handle* h, gpp_timings* out);
int gpp_get_stats(gpp_handle* h, gpp_stats* out);

/* dense K (without noise) of the training inputs, k_out is [n*n] row-major
 * (covar_module(x).evaluate(), models/gp_plus.py:472-474) */
int gpp_covariance(gpp_handle* h, const gpp_hyper* hyper, double* k_out);

/* debugging / parity probes: copy the factor L (lower, [n*n]), its inverse, or K_y^{-1} of the
 * last evaluation back to the host.  which: 0 = L, 1 = L^{-1}, 2 = K_y^{-1}, 3 = alpha ([n]),
 * 4 = diag(K_y^{-1}) ([n]; needs an evaluation with gradient; loocv_rrmse, optim/mll_noise_continuation.py:28-42) */
int gpp_fetch(gpp_handle* h, int which, double* out);

/* prediction: factorize once for fixed hyper-parameters (DefaultPredictionStrategy cache,
 * models/gpregression.py:126-131), then stream candidates */
int gpp_factorize(gpp_handle* h, const gpp_hyper* hyper);

/* mean[m], var[m] in SCALED y units (the caller applies y_min/y_std, gpregression.py:142-147).
 * noise_idx: per-candidate noise group used when include_noise != 0 (gpregression.py:136-140).
 * var is clamped below at min_var (gpytorch min_variance, 1e-10 in double). */
int gpp_predict(gpp_handle* h, int64_t m, const double* xq, const int32_t* level_idx,
                const int32_t* noise_idx, const int32_t* mean_idx, int include_noise,
                double min_var, double* mean, double* var);

/* GP_Plus.predict_with_grad (models/gp_plus.py:626-628): gpp_predict plus, per candidate, the derivatives of the
 * scaled mean and of the clamped variance w.r.t. its quantitative inputs xq; d_mean, d_var are [m*dq] row-major,
 * either may be NULL.  mean/var are bitwise those of gpp_predict.  Same pointer conventions as gpp_predict.
 * d_var is 0 where the variance was clamped at min_var; categorical / source inputs have no derivative. */
int gpp_predict_grad(gpp_handle* h, int64_t m, const double* xq, const int32_t* level_idx,
                     const int32_t* noise_idx, const int32_t* mean_idx, int include_noise, double min_var,
                     double* mean, double* var, double* d_mean, double* d_var);

/* Joint posterior over m <= GPP_MAX_JOINT candidates: the full predictive covariance
 *   Sigma* = K** - K* K_y^-1 K*^T  (+ noise of each candidate's group on the diagonal when include_noise)
 * and draws from N(mean, Sigma*).  Replace GPR.posterior's joint GPyTorchPosterior (gpregression.py:151-166) and
 * the MultivariateNormal.rsample of gpytorch that its fantasize / samplers call (gpregression.py:177-221).
 * Same pointer conventions as gpp_predict (host or device, cudaMemcpyDefault).  Neither call changes the factor of
 * K_y, alpha, gpp_get_stats or gpp_get_timings: gpp_predict / gpp_fetch return bitwise the same afterwards.  The
 * candidate buffers (about 6 GiB at m = N = 16384) are allocated on the first call and freed with the handle;
 * gpp_sample_posterior adds one chunk of base samples and one of draws, min(n_samples, 2^27/m) rows each (up to
 * 2 x 1 GiB), so up to about 8 GiB at m = N = 16384.  m > GPP_MAX_JOINT returns GPP_ERR_ARG before any
 * allocation. */
#define GPP_MAX_JOINT 16384

/* mean[m] (bitwise gpp_predict's), cov[m*m] row-major, exactly symmetric, scaled y units, NOT clamped.
 * Either output may be NULL. */
int gpp_predict_joint(gpp_handle* h, int64_t m, const double* xq, const int32_t* level_idx,
                      const int32_t* noise_idx, const int32_t* mean_idx, int include_noise,
                      double* mean, double* cov);

/* samples[s*m+i] = mean_i + sum_j L[i,j] base_samples[s*m+j],  L L^T = cov + jitter*I (psd_safe_cholesky ladder:
 * jitter 0, 1e-8, 1e-7, 1e-6; the one that succeeded is written to *jitter, GPP_ERR_NOT_PD when none does).
 * base_samples and samples are [n_samples*m] row-major; with base_samples = I_m the draws are mean + L^T rows. */
int gpp_sample_posterior(gpp_handle* h, int64_t m, const double* xq, const int32_t* level_idx,
                         const int32_t* noise_idx, const int32_t* mean_idx, int include_noise,
                         int64_t n_samples, const double* base_samples, double* samples, double* jitter);

/* Joint posteriors of b independent t-batches of q candidates each (Monte-Carlo batch acquisition: qEI, qNEI, qUCB
 * and qKG call posterior on a [b, q, d] batch).  Same pointer conventions as gpp_predict (host or device,
 * cudaMemcpyDefault).  Only the q x q diagonal blocks are formed, so the cost over gpp_predict at the same b*q rows is
 * about q/N for the covariance and the same for its gradient over gpp_predict_grad.  Neither call changes the factor
 * of K_y, alpha, gpp_get_stats or gpp_get_timings.  The chunk buffers are those of gpp_predict_grad plus one chunk's
 * q x q blocks, allocated on the first call and freed with the handle.  q > GPP_MAX_QBATCH, q < 1, b < 0 or dq > 32
 * return GPP_ERR_ARG before any allocation. */
#define GPP_MAX_QBATCH 128   /* q: points per t-batch, at most one 128-row tile */

/* Mean and joint covariance of each of b independent t-batches of q candidates.
 * Candidate rows are t-batch-major: xq is [b*q*dq], and level_idx / noise_idx / mean_idx are [b*q].
 * Outputs, in scaled units:
 *   mean [b*q]    bitwise gpp_predict's at the same rows
 *   cov  [b*q*q]  Sigma_t = K**_t - K*_t K_y^-1 K*_t^T (+ each row's noise when include_noise)
 * cov is exactly symmetric and not clamped. Its diagonal is bitwise the unclamped variance that gpp_predict forms
 * from the same row sums, sf2 - sum_t rowsq[t][i] (+ noise_i), before the min_var clamp.  A t-batch's outputs do not
 * depend on the other t-batches of the call.  Either output may be NULL. */
int gpp_posterior_qbatch(gpp_handle* h, int64_t b, int32_t q, const double* xq, const int32_t* level_idx,
                         const int32_t* noise_idx, const int32_t* mean_idx, int include_noise,
                         double* mean, double* cov);

/* Vector-Jacobian product of gpp_posterior_qbatch at the same arguments.
 * Inputs:  g_mean [b*q], g_cov [b*q*q], both upstream gradients; either may be NULL (zero).
 * Output:  d_xq [b*q*dq] = d/d xq of ( sum g_mean*mean + sum g_cov*cov ), quantitative inputs only. */
int gpp_posterior_qbatch_grad(gpp_handle* h, int64_t b, int32_t q, const double* xq, const int32_t* level_idx,
                              const int32_t* noise_idx, const int32_t* mean_idx, int include_noise,
                              const double* g_mean, const double* g_cov, double* d_xq);

/* Monte-Carlo batch acquisition of b t-batches of q_tot rows (botorch's qEI, qNEI, qUCB with base samples shared by
 * every t-batch), and its gradient in xq.  Pointer conventions as gpp_posterior_qbatch (host or device,
 * cudaMemcpyDefault).  Per t-batch t, with mu_t and Sigma_t bitwise gpp_posterior_qbatch's (scaled units):
 *   L_t = chol(Sigma_t + j_t I), j_t the first of 0, 1e-8, 1e-7, 1e-6 whose pivots are all > 0
 *   y_s = mu_t + L_t e_s for each base-sample row e_s, sigma = +1 when maximize, -1 otherwise
 *   values[t] = (1/S) sum_s u(y_s) with u
 *     GPP_QACQ_EI   max(max_i sigma y_si - sigma best_f, 0)                          (n_baseline = 0)
 *     GPP_QACQ_NEI  max(max_{i<q} sigma y_si - max_{q<=j<q_tot} sigma y_sj, 0)      (the last n_baseline rows of each
 *                   t-batch are baseline points, q = q_tot - n_baseline, 1 <= n_baseline < q_tot)
 *     GPP_QACQ_UCB  max_i (sigma mu_i + sqrt(beta pi / 2) |y_si - mu_i|)            (n_baseline = 0, beta >= 0)
 *   d_xq [b*q_tot*dq] = d(sum_t values[t]) / d xq over all q_tot rows, quantitative inputs only (NULL: values only)
 *   jitter [b] = j_t (may be NULL)
 * A t-batch's outputs do not depend on the other t-batches of the call.  The call does not change the factor of K_y,
 * alpha, gpp_get_stats or gpp_get_timings.  GPP_ERR_NOT_PD when a t-batch fails every rung, GPP_ERR_NAN on NaN.  An
 * unknown kind, n_baseline out of range for the kind, q_tot outside [1, GPP_MAX_QBATCH], n_samples outside
 * [1, GPP_MAX_MC_SAMPLES], a missing base_samples or values, or dq > 32 return GPP_ERR_ARG before any allocation.
 * The base samples (n_samples*q_tot doubles) and one chunk's values and jitters are held on the device from the first
 * call and freed with the handle. */
#define GPP_QACQ_EI 0
#define GPP_QACQ_NEI 1
#define GPP_QACQ_UCB 2
#define GPP_MAX_MC_SAMPLES 65536
int gpp_acq_qbatch(gpp_handle* h, int64_t b, int32_t q_tot, const double* xq, const int32_t* level_idx,
                   const int32_t* noise_idx, const int32_t* mean_idx, int include_noise,
                   int kind, int32_t n_baseline, double best_f, double beta, int maximize,
                   int64_t n_samples, const double* base_samples,   /* [n_samples * q_tot], shared by all t-batches */
                   double* values,                                  /* [b] */
                   double* d_xq,                                    /* [b * q_tot * dq] or NULL: values only */
                   double* jitter);                                 /* [b] or NULL */

/* Batch integrated posterior variance (botorch's qNegIntegratedPosteriorVariance, acquisition/active_learning.py:
 * qNegIntegratedPosteriorVariance.forward, which averages posterior(mc_points).variance of
 * model.fantasize(X_t, observation_noise=True) over the integration points).  The fantasised variance does not depend
 * on the fantasised y, so the engine evaluates the closed form below; all quantities are in scaled y units.
 *
 * gpp_ipv_points stores the integration set X_I of m points (1 <= m <= GPP_MAX_IPV_POINTS) on the handle: its point
 * panels, U_I = K(X_I, X) L^-T, V_I = U_I L^-1 and vbar = (1/m) sum_m v_m with v_m = sf2 - |U_m|^2 (gpp_predict's
 * variance without noise or clamp).  Pointer conventions as gpp_predict (host or device, cudaMemcpyDefault).  The set
 * stays valid until the factor or the hyper-parameters of the handle change (gpp_factorize, gpp_mll_grad, the
 * gpp_objective calls, gpp_covariance); it then has to be stored again.  It takes [mp x Np] doubles twice (mp = m
 * rounded up to 128) plus the panels, held from the first call and freed with the handle.
 *
 * gpp_nipv_qbatch evaluates b t-batches of q rows against the stored set.  Per t-batch t, with Sigma_t bitwise
 * gpp_posterior_qbatch's:
 *   C_t = K(X_I, X_t) - U_I U_t^T                                    [m x q] posterior cross-covariance
 *   A_t = Sigma_t + diag(noise of each row's group) + j_t I         j_t the first of 0, 1e-8, 1e-7, 1e-6 that factors
 *   values[t] = -vbar + (1/m) tr(A_t^-1 C_t^T C_t)                   minus the mean posterior variance over X_I after
 *                                                                    also observing X_t
 *   d_xq [b*q*dq] = d(sum_t values[t]) / d xq, quantitative inputs only (NULL: values only)
 *   jitter [b] = j_t (may be NULL)
 * A t-batch's outputs do not depend on the other t-batches of the call or on how it is split into chunks.  The call
 * does not change the factor of K_y, alpha, gpp_get_stats or gpp_get_timings.  GPP_ERR_NOT_PD when a t-batch fails
 * every rung, GPP_ERR_NAN on NaN.  No valid integration set, q outside [1, GPP_MAX_QBATCH], b < 0, a missing values
 * or dq > 32 return GPP_ERR_ARG before any allocation.  One chunk's C^T (at most 1 GiB), q x q blocks and gradient
 * partials are held on the device from the first call and freed with the handle. */
#define GPP_MAX_IPV_POINTS 16384
int gpp_ipv_points(gpp_handle* h, int64_t m, const double* xq, const int32_t* level_idx);
int gpp_nipv_qbatch(gpp_handle* h, int64_t b, int32_t q, const double* xq, const int32_t* level_idx,
                    const int32_t* noise_idx,
                    double* values,   /* [b] */
                    double* d_xq,     /* [b * q * dq] or NULL: values only */
                    double* jitter);  /* [b] or NULL */

/* One-shot knowledge gradient (botorch's qKnowledgeGradient.forward, acquisition/knowledge_gradient.py, with the
 * PosteriorMean value function and current_value = None).  Each of the b t-batches holds q_tot = q + n_fantasies
 * consecutive rows of xq: the q actual points X_t, then the F = n_fantasies fantasy solutions x'_f (botorch's
 * X_actual_and_fantasies layout, _split_fantasy_points).  With mu and Sigma bitwise those of
 * gpp_posterior_qbatch(..., include_noise = 1) on the same rows (a NULL noise_idx means group 0), in scaled y units:
 *   A_t = Sigma[0:q, 0:q] + j_t I,  L_t = chol(A_t)   j_t the first of 0, 1e-8, 1e-7, 1e-6 that factors
 *   c_f = Sigma[0:q, q+f]                             posterior cross-covariance of X_t and x'_f
 *   values[t] = (1/F) sum_f sigma (mu[q+f] + (L_t^-1 c_f) . e_f)   sigma = +1 to maximise, -1 to minimise
 * e_f is row f of base_samples [F x q], shared by every t-batch.  Each term is the posterior mean at x'_f of the model
 * that also observed X_t, each row with its group's noise, at y_f = mu[0:q] + L_t e_f.
 *   d_xq [b*q_tot*dq] = d(sum_t values[t]) / d xq for all q_tot rows, quantitative inputs only (NULL: values only)
 *   jitter [b] = j_t (may be NULL)
 * A t-batch's outputs do not depend on the other t-batches of the call or on how it is split into chunks.  The call
 * does not change the factor of K_y, alpha, gpp_get_stats or gpp_get_timings.  GPP_ERR_NOT_PD when a t-batch fails
 * every rung, GPP_ERR_NAN on NaN.  q < 1, n_fantasies < 1, q + n_fantasies > GPP_MAX_QBATCH, b < 0, a missing
 * base_samples or values, or dq > 32 return GPP_ERR_ARG before any allocation.  It uses the buffers of gpp_acq_qbatch
 * and allocates none of its own. */
int gpp_kg_qbatch(gpp_handle* h, int64_t b, int32_t q, int32_t n_fantasies, const double* xq,
                  const int32_t* level_idx, const int32_t* noise_idx, const int32_t* mean_idx, int maximize,
                  const double* base_samples,  /* [n_fantasies * q], shared by all t-batches */
                  double* values,              /* [b] */
                  double* d_xq,                /* [b * (q + n_fantasies) * dq] or NULL: values only */
                  double* jitter);             /* [b] or NULL */

/* GIBBON, the lower bound of max-value entropy search (botorch's qLowerBoundMaxValueEntropy and, with target rows,
 * qMultiFidelityLowerBoundMaxValueEntropy, acquisition/max_value_entropy_search.py; Moss et al., 2021).  Each of the b
 * t-batches holds q_tot consecutive rows of xq: the q actual points x_1..x_q, then with projected = 1 their copies
 * g_1..g_q at the target fidelity (tau(i) = q + i, q_tot = 2q; projected = 0: tau(i) = i, q_tot = q).  With mu and
 * Sigma bitwise those of gpp_posterior_qbatch(..., include_noise = 0) on the same rows, n_i the noise of row i's group
 * (a NULL noise_idx means group 0), eps = 1e-8, sigma = +1 to maximise and -1 to minimise, in scaled y units:
 *   V = Sigma[0:q, 0:q] + diag(n_i),  L L^T = V + j_t I   j_t the first of 0, 1e-8, 1e-7, 1e-6 that factors
 *   v_i = max(V_ii, eps)  s_i^2 = max(Sigma_tau(i)tau(i), eps)  c_i = Sigma_i,tau(i)  rho_i^2 = c_i^2 / (v_i s_i^2)
 *   gamma_ik = (m_k - sigma mu_tau(i)) / s_i,  r_ik = phi(gamma_ik) / max(Phi(gamma_ik), eps)
 *   Q_i = -(1/2K) sum_k log max(1 - rho_i^2 r_ik (gamma_ik + r_ik), eps)      quality of row i
 *   D   = sum_i (log L_ii - 1/2 log (V + j_t I)_ii)                            diversity
 *   values[t] = D + sum_i Q_i   (nats)
 * m_k = max_values[k], K = n_max_values samples of max sigma f in scaled units, shared by every t-batch.
 *   d_xq [b*q_tot*dq] = d(sum_t values[t]) / d xq for all q_tot rows, quantitative inputs only (NULL: values only)
 *   jitter [b] = j_t (may be NULL)
 * A t-batch's outputs do not depend on the other t-batches of the call or on how it is split into chunks.  The call
 * does not change the factor of K_y, alpha, gpp_get_stats or gpp_get_timings.  GPP_ERR_NOT_PD when a t-batch fails
 * every rung, GPP_ERR_NAN on NaN.  q < 1, projected not 0 or 1, q_tot > GPP_MAX_QBATCH, b < 0, n_max_values outside
 * [1, GPP_MAX_MC_SAMPLES], a missing max_values or values, or dq > 32 return GPP_ERR_ARG before any allocation.  It
 * uses the buffers of gpp_acq_qbatch (the max values in its base-sample buffer) and allocates none of its own. */
int gpp_gibbon_qbatch(gpp_handle* h, int64_t b, int32_t q, int32_t projected, const double* xq,
                      const int32_t* level_idx, const int32_t* noise_idx, const int32_t* mean_idx, int maximize,
                      int64_t n_max_values, const double* max_values, /* [K] samples of max sigma f, scaled units */
                      double* values,                               /* [b] */
                      double* d_xq,                                 /* [b * q_tot * dq] or NULL: values only */
                      double* jitter);                              /* [b] or NULL */

/* Quartiles of the maximum of sigma f over m candidates under independent marginals (botorch's
 * _sample_max_value_Gumbel, acquisition/max_value_entropy_search.py, without the marginals leaving the device).  The
 * marginals mu_j, s_j^2 are gpp_predict's at include_noise = 0, min_var = 1e-8 (bitwise), held in two buffers of m
 * doubles on the handle.  quartiles[0..2] solve l(y) = sum_j log Phi((y - sigma mu_j) / s_j) = log p for p = 1/4, 1/2,
 * 3/4 by bisection, each to within 1e-12 (hi - lo) of the bracket: lo = min sigma mu - 5 max s, hi = max sigma mu +
 * 5 max s, hi doubled away from lo while l(hi) < log 3/4.  The sums run in an order that depends only on m.  GPP_ERR_NAN
 * on a NaN or infinite marginal; m < 1, a missing quartiles, xq or level_idx, or dq > 32 return GPP_ERR_ARG.  quartiles may be
 * host or device memory. */
int gpp_max_value_quartiles(gpp_handle* h, int64_t m, const double* xq, const int32_t* level_idx,
                            const int32_t* mean_idx, int maximize, double* quartiles /* [3], scaled units */);

/* fused predict + acquisition + argmax over m candidates (BO_GP_plus.py:183-194).
 * y_min/y_std undo the target scaling; cost_idx[m] selects cost[n_cost]; kind_by_cost[n_cost]
 * selects GPP_ACQ_* per source (HF for source 0, LF otherwise in the reference).
 * best_f[n_cost] is the incumbent per source.  Returns the best score and its index
 * (first index on ties, like torch.argmax). scores may be NULL or [m]. */
int gpp_acq_argmax(gpp_handle* h, int64_t m, const double* xq, const int32_t* level_idx,
                   const int32_t* mean_idx, const int32_t* cost_idx, int32_t n_cost,
                   const double* cost, const int32_t* kind_by_cost, const double* best_f,
                   int maximize, double si, double y_min, double y_std, double min_var,
                   double* scores, double* best_score, int64_t* best_index);

/* ---- the O(p) host side of MLLObjective.fun inside the library --------------------------------
 * gpp_objective(theta) = -( log N(y; m, K_y) + sum log-priors ) and its gradient w.r.t. the RAW parameter
 * vector theta that scipy optimises -- the whole body of MLLObjective.fun (optim/mll_scipy.py:112-127:
 * float32 cast of theta :97, raw->natural transforms, marginal_log_likelihood :37-47, backward :123,
 * pack_grads :101-110) in one call that holds no Python lock.  The layout is compiled from the model by
 * gpplus_b200/optim/_fast_objective.py and checked there against the torch path.
 *   ls_kind 0: lengthscale = exp(raw) (gpytorch Positive(exp));  1: 2^-1/2 * 10^(-raw/2) (models/gp_plus.py:252)
 *   w_num 0.5 / 1.0: w = w_num / lengthscale^2 (RBF / Matern families);  0: w = lengthscale (kernels/Rough_RBF.py)
 * Offsets index theta; a negative offset means "frozen": the *_const value is used and no gradient is written. */
#define GPP_PRIOR_NORMAL 0        /* raw parameters:   a = loc[len], b = scale[len]                      */
#define GPP_PRIOR_LOGNORMAL_OS 1  /* CONSTRAINED outputscale (gpregression.py:113-115): a[0]=loc, b[0]=scale */
#define GPP_PRIOR_HORSESHOE 2     /* raw noise:        a = scale[len], b = lb[len]  (priors/horseshoe.py:60-66) */
#define GPP_PRIOR_MOLLIFIED 3     /* raw lengthscale:  a = lo[len], b = hi[len], c = tail_sigma[len]       */
#define GPP_PRIOR_CONST 4         /* frozen parameter: a[0] = its constant log-density                     */

typedef struct gpp_prior {
    int32_t kind, off, len;
    const double *a, *b, *c;
} gpp_prior;

typedef struct gpp_theta_layout {
    int32_t p;                  /* length of theta */
    int32_t off_latent;         /* A [dz x n_onehot] row-major (nn.Linear weight, models/gp_plus.py:1245-1247) */
    int32_t n_onehot;
    const double* zeta;         /* [n_combo x n_onehot] one-hot table (models/gp_plus.py:1027-1073) */
    const double* latent_const; /* [dz x n_onehot] when off_latent < 0 */
    double latent_ls;           /* fixed lengthscale of the latent RBF kernel (models/gp_plus.py:223-226) */
    int32_t off_noise;          /* raw_noise [n_noise]; noise = noise_lb + exp(raw) */
    const double* noise_const;
    double noise_lb;
    int32_t off_os;             /* raw_outputscale; sigma_f^2 = softplus(raw) */
    double os_const;
    int32_t off_ls;             /* raw_lengthscale [dq] */
    const double* ls_const;
    int32_t ls_kind;
    double w_num;
    const int32_t* off_mean;    /* [n_mean] offsets of the mean constants */
    const double* mean_const;   /* [n_mean] */
    int32_t n_priors;
    const gpp_prior* priors;    /* evaluated in this order (named_priors order) */
} gpp_theta_layout;

/* copies the layout (and every array it points to) into the handle */
int gpp_set_theta_layout(gpp_handle* h, const gpp_theta_layout* layout);
/* value = neg log posterior at theta[p]; grad[p] may be NULL when want_grad == 0; detail may be NULL */
int gpp_objective(gpp_handle* h, const double* theta, int want_grad, double* value, double* grad,
                  gpp_mll_result* detail);

/* Split form for callers that keep many handles in flight from ONE host thread (the lock-step multi-start driver
 * behind fit_model_scipy, optim/mll_scipy.py:287-293 of the reference fans restarts out over processes):
 * gpp_objective_enqueue issues the evaluation on the handle's stream and returns without waiting;
 * gpp_objective_collect waits for it, walks the rest of the jitter ladder if needed, and returns exactly what
 * gpp_objective would have returned (want_grad as given to enqueue). */
int gpp_objective_enqueue(gpp_handle* h, const double* theta, int want_grad);
int gpp_objective_collect(gpp_handle* h, double* value, double* grad, gpp_mll_result* detail);

/* Arithmetic of the three O(N^3) stages (factorisation trailing updates, triangular inverse, K^-1).  Both produce
 * FP64 results within the parity tolerances (objective 1e-9, gradient 1e-8; observed 2e-13 / 3e-13 at N = 16384):
 *   GPP_FP64_DMMA  mma.sync FP64 tensor-core tiles (IEEE FP64 products and sums)
 *   GPP_FP64_INT8  operands cut into 7 signed base-256 digit planes per power-of-two-scaled row, exact integer products
 *                  on the INT8 tcgen05 tensor cores, FP64 recombination (csrc/oz_gemm.cuh).  Default from N = 3072.
 * gpp_set_fp64_mode sets the process-wide choice for handles created afterwards (-1 = by size, the default;
 * the environment variable GPP_FP64=dmma has the same effect as 0) and returns the previous one;
 * gpp_get_fp64_mode reports what a handle uses. */
#define GPP_FP64_DMMA 0
#define GPP_FP64_INT8 1
int gpp_set_fp64_mode(int mode);
int gpp_get_fp64_mode(gpp_handle* h);

/* raw issue rate of tcgen05.mma kind::i8 (M = 128, N = n_cols in {64, 128, 256}) on resident operands, whole GPU,
 * in int8 tera-ops per second: the roofline denominator of the INT8-sliced path (bench.py measures it live) */
int gpp_probe_i8(int device, int n_cols, int iters, double* tops_out);

/* FP64 DMMA GEMM probe used by bench/selftest: C[m x n] = A[m x k] * B[n x k]^T on device
 * scratch, returns average milliseconds per launch over iters (m,n,k multiples of 128). */
int gpp_probe_dgemm(int device, int m, int n, int k, int iters, float* ms_out);

#ifdef __cplusplus
}
#endif
#endif /* GPPLUS_B200_H */
