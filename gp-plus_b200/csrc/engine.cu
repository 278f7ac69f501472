// C-ABI engine: exact-GP MLL + gradient, factorisation, batched prediction and acquisition arg-max
// on one B200 (sm_100a).  Entry points are declared (with the reference call sites they replace) in
// include/gpplus_b200.h.  There is no CPU fallback anywhere in this file.
#include "../../include/gpplus_b200.h"

#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <mutex>
#include <string>
#include <vector>

#include "chol.cuh"
#include "cov.cuh"
#include "gibbon.cuh"
#include "joint.cuh"
#include "kg.cuh"
#include "objective.h"
#include "predict.cuh"
#include "predict_grad.cuh"
#include "nipv.cuh"
#include "qacq.cuh"
#include "qbatch.cuh"
#include "solve.cuh"

using namespace gpp;

static thread_local std::string g_err;

static void set_err(const char* what, cudaError_t e) {
    char buf[512];
    snprintf(buf, sizeof(buf), "%s: %s (%s)", what, cudaGetErrorName(e), cudaGetErrorString(e));
    g_err = buf;
}

#define CK(x)                         \
    do {                              \
        cudaError_t e_ = (x);         \
        if (e_ != cudaSuccess) {      \
            set_err(#x, e_);          \
            return GPP_ERR_CUDA;      \
        }                             \
    } while (0)

#define ARG_FAIL(msg)       \
    do {                    \
        g_err = msg;        \
        return GPP_ERR_ARG; \
    } while (0)

enum { EV_START = 0, EV_COV, EV_CHOL, EV_TRTRI, EV_SOLVE, EV_LAUUM, EV_GRAD, EV_END, EV_COUNT };

// Everything gpp_create decides besides the problem's shape: the arithmetic of the O(N^3) stages (gpp_set_fp64_mode,
// GPP_FP64) and the schedule switches of the handle (int fields only: compared with memcmp).  A parked handle is
// handed back only when the configuration in force now equals the one it was built under.
struct CreateConfig {
    int lookahead = 1;     // look-ahead / lazy-panel factorisation; GPP_CHOL=blocked: potrf_blocked
    int graph = 0;         // CUDA-graph replay of a whole evaluation (GPP_GRAPH)
    int small_block = 0;   // T <= 16: CTAs of the one-launch factorisation (GPP_SMALL_BLOCK; 0 = launch chain)
    int int8 = 0;          // INT8-sliced O(N^3) stages
    CholSchedule chol;
    OzSchedule oz;         // used when the handle carries an OzCtx
};

template <typename Tp>
static cudaError_t dev_alloc(Tp** p, size_t count) {
    return cudaMalloc((void**)p, std::max<size_t>(count, 1) * sizeof(Tp));
}

// Grow-only device array of the prediction workspace, allocated on first use.  reserve() keeps the storage when it
// holds `count` elements already; otherwise it waits for the stream, frees the storage and allocates `count` elements,
// zero-filled when asked.  The storage is freed with the array, i.e. with the handle.
template <typename Tp>
struct DevArray {
    Tp* p = nullptr;
    size_t cap = 0;  // elements
    DevArray() = default;
    DevArray(const DevArray&) = delete;
    DevArray& operator=(const DevArray&) = delete;
    ~DevArray() { release(); }
    operator Tp*() const { return p; }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
    cudaError_t reserve(long long count, cudaStream_t st, bool zero = false) {
        if (count <= (long long)cap) return cudaSuccess;
        cudaError_t e = cudaStreamSynchronize(st);
        if (e != cudaSuccess) return e;
        release();
        if ((e = dev_alloc(&p, (size_t)count)) != cudaSuccess) {
            p = nullptr;
            return e;
        }
        cap = (size_t)count;
        return zero ? cudaMemsetAsync(p, 0, sizeof(Tp) * (size_t)count, st) : cudaSuccess;
    }
};

// Candidate points kept on the handle between calls (the joint set, the integration set): their inputs and prepared
// panels, m points padded to mp rows, and U = K* L^-T [mp x Np] (load_point_set)
struct PointSet {
    long long mp = 0;  // rows of the set last loaded (the panels' leading dimension)
    DevArray<double> xq, xs, nrm, zpt, U;
    DevArray<int> lvl;
};

struct gpp_handle {
    int device = 0;
    cudaStream_t st = nullptr;
    long long n = 0, np = 0;
    int T = 0;
    int dq = 0, dqp = 0, dz = 0, n_combo = 0, n_noise = 0, n_mean = 0, kernel = 0;
    int n_pass = 1;  // latent tables averaged into K (multi-pass ensemble covariance, gp_plus.py:387-399)
    // static training data
    double *xq = nullptr, *y = nullptr, *centre = nullptr;
    int *level_idx = nullptr, *noise_idx = nullptr, *mean_idx = nullptr;
    // hyper-parameters (device copy): [w dq | ztab n_pass*n_combo*dz | noise | beta]
    double* hyp = nullptr;
    double* hyp_host = nullptr;  // pinned
    int hyp_len = 0;
    double sf2 = 0.0;
    // per-evaluation point panels
    double *xs = nullptr, *xst = nullptr, *nrm = nullptr, *zpt = nullptr, *r = nullptr, *diag_add = nullptr;
    double *v = nullptr, *alpha = nullptr, *part = nullptr;
    // N x N work matrices
    double *A = nullptr, *M = nullptr, *S = nullptr;
    double* logdet_part = nullptr;
    int* info = nullptr;
    int* info_host = nullptr;  // pinned
    double *tile_part = nullptr, *zpart = nullptr, *gz = nullptr;
    double* res = nullptr;
    double* res_host = nullptr;  // pinned
    double* gz_host = nullptr;   // pinned
    int res_len = 0;
    std::vector<int> level_idx_host;
    // prediction workspace (DESIGN.md §3).  Chunk buffers of mc_alloc rows (their leading dimension):
    long long mc_alloc = 0;
    DevArray<double> c_xq, c_xs, c_nrm, c_zpt, c_K, c_mean_part, c_rowsq, c_mu, c_var, c_score, c_blk_best;
    DevArray<int> c_lvl, c_noise, c_mean, c_cost;
    DevArray<long long> c_blk_idx;
    DevArray<double> acq_par;  // gpp_acq_argmax: [cost n_cost | best_f n_cost]
    DevArray<int> acq_kind;
    // gradient and t-batch paths: chunks of g_step rows with U = K* L^-T stored, the gradient partials and results
    long long g_step = 0;
    DevArray<double> g_U, g_part_m, g_part_v, g_dmean, g_dvar;
    // t-batch paths: one chunk's q x q blocks (Sigma out, or the upstream gradient G in) and its upstream mean gradient
    DevArray<double> q_buf, q_gm;
    // gpp_acq_qbatch / gpp_nipv_qbatch / gpp_kg_qbatch / gpp_gibbon_qbatch: the base samples (max values) of the call,
    // one chunk's values and jitters, the status word
    DevArray<double> a_E, a_val, a_jit;
    DevArray<int> a_info;
    // gpp_max_value_quartiles: the m marginal means and variances, the per-block partials, the bracket state and the
    // NaN flag
    DevArray<double> v_mu, v_var, v_part, v_state;
    DevArray<int> v_nan;
    // gpp_predict_joint / gpp_sample_posterior: the joint set and, ld the call's mp, Sigma* (then L*), the diagonal-block
    // inverses of L* (a full [mp x mp] matrix: potrf_blocked addresses them with Sigma*'s leading dimension), the
    // diagonal additions, mu, the log-determinant partials, the noise groups, the status word, and one chunk of base
    // samples and draws
    PointSet jset;
    DevArray<double> j_S, j_Minv, j_diag, j_mu, j_logdet, j_E, j_Y;
    DevArray<int> j_noise, j_info;
    // integration set of gpp_nipv_qbatch (gpp_ipv_points): i_m points, V_I = U_I L^-1 [mp x Np], a zero vector in the
    // place of alpha, the mean latent variance, and the factor generation the set was built for
    PointSet iset;
    long long i_m = 0, i_gen = -1;
    double i_vbar = 0.0;
    DevArray<double> i_V, i_zero;
    // gpp_nipv_qbatch chunks: C^T [rows x mp of the set], the Gram and A^-1 blocks, and the gradient partials over the
    // training and the integration column tiles
    DevArray<double> n_C, n_G, n_Ai, n_pm, n_pv;
    long long fgen = 0;  // bumped whenever the factor (or its hyper-parameters) changes
    bool factorized = false;
    double last_jitter = 0.0;
    cudaEvent_t ev[EV_COUNT];
    bool ev_valid[EV_COUNT];
    gpp_timings tm;
    CholLookahead la;
    OzCtx* oz = nullptr;     // INT8-sliced tcgen05 path of the O(N^3) stages (large problems; GPP_FP64=dmma turns it off)
    // CUDA-graph replay of one whole evaluation (small problems are launch-bound): [want_grad]
    cudaGraphExec_t graph_exec[2] = {nullptr, nullptr};
    long long graph_kernels[2] = {0, 0};
    bool use_graph = false;  // cfg.graph until a capture fails
    bool capturing = false;
    bool pending = false;    // gpp_objective_enqueue issued, gpp_objective_collect not yet called
    int pending_grad = 0;
    void* slab = nullptr;         // one device allocation holds every per-handle buffer below (gpp_create)
    size_t slab_bytes = 0;
    int* idx_slots[3] = {nullptr, nullptr, nullptr};  // storage of level_idx / noise_idx / mean_idx inside the slab
    void* pinned_slab = nullptr;  // one pinned allocation holds hyp_host / info_host / res_host / gz_host
    gpp_stats stats;
    cudaEvent_t ev_info = nullptr;                 // factorisation status available (jitter-ladder early-out)
    ThetaLayout layout;                            // optional: O(p) host side of MLLObjective.fun
    std::vector<double> g_w, g_z, g_noise, g_beta;  // gradient scratch of gpp_objective
    CreateConfig cfg;                              // configuration the handle was created under
};

static const double* hyp_w(const gpp_handle* h) { return h->hyp; }
static const double* hyp_z(const gpp_handle* h) { return h->hyp + h->dq; }
static int ztab_len(const gpp_handle* h) { return h->n_pass * h->n_combo * h->dz; }
static const double* hyp_noise(const gpp_handle* h) { return h->hyp + h->dq + ztab_len(h); }
static const double* hyp_beta(const gpp_handle* h) { return h->hyp + h->dq + ztab_len(h) + h->n_noise; }
// per-evaluation scalars live behind the vectors so that graph replays need no new kernel arguments
static const double* hyp_sf2(const gpp_handle* h) { return hyp_beta(h) + h->n_mean; }
static const double* hyp_jitter(const gpp_handle* h) { return hyp_beta(h) + h->n_mean + 1; }

extern "C" int gpp_version(void) { return 113; }

// process-wide default for handles created afterwards: -1 = by size (INT8-sliced from Np = 4096), 0 = DMMA, 1 = INT8
static std::atomic<int> g_fp64_mode{-1};
extern "C" int gpp_set_fp64_mode(int mode) {
    if (mode < -1 || mode > 1) return g_fp64_mode.load();
    return g_fp64_mode.exchange(mode);
}
extern "C" int gpp_get_fp64_mode(gpp_handle* h) { return (h && h->oz && h->oz->ready) ? GPP_FP64_INT8 : GPP_FP64_DMMA; }

extern "C" int gpp_device_count(void) {
    int c = 0;
    if (cudaGetDeviceCount(&c) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return c;
}

extern "C" const char* gpp_last_error(void) { return g_err.c_str(); }

extern "C" long long gpp_launch_count(void) { return g_launches.load(); }

static void destroy_now(gpp_handle* h) {
    if (!h) return;
    cudaSetDevice(h->device);
    if (h->st) cudaStreamSynchronize(h->st);
    if (h->slab) cudaFree(h->slab);
    if (h->pinned_slab) cudaFreeHost(h->pinned_slab);
    for (int i = 0; i < EV_COUNT; i++) cudaEventDestroy(h->ev[i]);
    if (h->ev_info) cudaEventDestroy(h->ev_info);
    for (int i = 0; i < 2; i++)
        if (h->graph_exec[i]) cudaGraphExecDestroy(h->graph_exec[i]);
    h->la.destroy();
    if (h->oz) {
        h->oz->destroy();
        delete h->oz;
    }
    if (h->st) cudaStreamDestroy(h->st);
    delete h;
}

// ---------------------------------------------------------------------------------------------
// Handle pool.  Creating a handle costs one cudaMalloc + one cudaMallocHost + three streams + a dozen events + two
// CUDA-graph instantiations, destroying it a synchronising cudaFree / cudaFreeHost: 5-25 ms each way on the GPU box,
// i.e. seconds for the 64 handles of a lock-step multi-start fit of a small model -- more than the fit itself.
// Released handles of small problems are therefore parked and handed back to the next gpp_create with the SAME
// shape on the same device (only the training data are re-uploaded; captured graphs stay valid because every
// device address and size is unchanged).  gpp_pool_clear() frees them.
static std::mutex g_pool_mu;
static std::vector<gpp_handle*> g_pool;
static size_t g_pool_bytes = 0;
static const size_t kPoolMaxHandleBytes = 192ull << 20;  // handles up to Np = 2816 (3 x Np^2 doubles)
static const size_t kPoolMaxBytes = 6ull << 30;
static const size_t kPoolMaxHandles = 160;

// the configuration a handle with T tile rows gets when it is created now: the production configuration, changed
// only by the environment variables set at this moment
static CreateConfig read_config(int T) {
    CreateConfig c;
    const char* e;
    if ((e = getenv("GPP_CHOL")) != nullptr) c.lookahead = strcmp(e, "blocked") != 0;
    c.graph = T <= 16;  // N <= 2048: an evaluation is a chain of ~25-100 tiny launches
    if ((e = getenv("GPP_GRAPH")) != nullptr) c.graph = atoi(e) != 0;
    if ((e = getenv("GPP_SMALL_BLOCK")) != nullptr) c.small_block = atoi(e);
    if ((e = getenv("GPP_PANEL")) != nullptr) c.chol.panel_blocks = atoi(e);
    if ((e = getenv("GPP_OVERLAP_INV")) != nullptr) c.chol.overlap_inverse = atoi(e);
    if ((e = getenv("GPP_BLOCK_CTAS")) != nullptr) c.chol.block_ctas = atoi(e);
    if ((e = getenv("GPP_TIMELINE")) != nullptr) c.chol.timeline = atoi(e) != 0;
    {
        // FP64 work of the O(N^3) stages: exact integer GEMMs on the INT8 tcgen05 tensor cores from Np = 3072 up
        // (measured: 3.08 vs 3.42 ms at N = 3072, 14.8 vs 22.0 at 8192, 28.8 vs 63.5 at 12288; below that an evaluation
        // is a CUDA-graph replay of latency-bound launches); GPP_FP64=dmma keeps everything on DMMA
        e = getenv("GPP_FP64");
        bool int8 = T >= 24;
        const int mode = g_fp64_mode.load();
        if (mode == GPP_FP64_DMMA) int8 = false;
        if (mode == GPP_FP64_INT8) int8 = T >= 8;   // forced: the stages still pick DMMA for shapes that are too small
        if (e && mode < 0) int8 = int8 && strcmp(e, "dmma") != 0;
        c.int8 = int8;
    }
    if (c.int8) {
        if ((e = getenv("GPP_OZ_MIN_TRAIL")) != nullptr) c.oz.min_trailing_tiles = atoi(e);
        if ((e = getenv("GPP_OZ_MIN_LEVEL")) != nullptr) c.oz.min_level_tiles = atoi(e);
        if ((e = getenv("GPP_OZ_NEXT")) != nullptr) c.oz.next_on_oz = atoi(e);
        if ((e = getenv("GPP_OZ_INNER")) != nullptr) c.oz.inner_min_k = atoi(e);
        if ((e = getenv("GPP_OZ_KINV_LEVELS")) != nullptr) c.oz.kinv_levels = atoi(e);
        if ((e = getenv("GPP_OZ_LAZY_MIN")) != nullptr) c.oz.lazy_min_tiles = atoi(e);
        if ((e = getenv("GPP_OZ_LAZY_PB")) != nullptr) c.oz.lazy_pb = std::min(std::max(atoi(e), 2), OzCtx::LAZY_PB);
        if ((e = getenv("GPP_OZ_STAGGER")) != nullptr) c.oz.stagger = atoi(e);
    }
    return c;
}

static bool same_shape(const gpp_handle* h, const gpp_problem* p, int device, const CreateConfig& cfg) {
    return memcmp(&h->cfg, &cfg, sizeof(cfg)) == 0 && h->device == device && h->n == p->n && h->dq == p->dq && h->dz == p->dz &&
           h->n_combo == (p->dz > 0 ? p->n_combo : 0) && h->n_noise == p->n_noise && h->n_mean == p->n_mean &&
           h->kernel == p->kernel && h->n_pass == (p->n_pass > 1 ? p->n_pass : 1) && (h->level_idx != nullptr) == (p->dz > 0 && p->level_idx != nullptr) &&
           (h->noise_idx != nullptr) == (p->noise_idx != nullptr) && (h->mean_idx != nullptr) == (p->mean_idx != nullptr);
}

extern "C" void gpp_pool_clear(void) {
    std::vector<gpp_handle*> victims;
    {
        std::lock_guard<std::mutex> lk(g_pool_mu);
        victims.swap(g_pool);
        g_pool_bytes = 0;
    }
    for (gpp_handle* h : victims) destroy_now(h);
}

extern "C" void gpp_destroy(gpp_handle* h) {
    if (!h) return;
    const char* e = getenv("GPP_POOL");
    const bool pooling = !(e && atoi(e) == 0);
    // a handle that has predicted (chunk or joint buffers allocated) is never parked
    if (pooling && h->slab_bytes <= kPoolMaxHandleBytes && h->mc_alloc == 0 && h->jset.mp == 0) {
        cudaSetDevice(h->device);
        if (h->st) cudaStreamSynchronize(h->st);
        std::lock_guard<std::mutex> lk(g_pool_mu);
        if (g_pool.size() < kPoolMaxHandles && g_pool_bytes + h->slab_bytes <= kPoolMaxBytes) {
            h->layout.set = false;
            h->factorized = false;
            h->fgen++;
            h->i_m = 0;
            h->pending = false;
            g_pool.push_back(h);
            g_pool_bytes += h->slab_bytes;
            return;
        }
    }
    destroy_now(h);
}

// training data of `p` into the (new or recycled) handle
static int upload_problem(gpp_handle* h, const gpp_problem* p) {
    const long long n = h->n;
    if (h->dq > 0) CK(cudaMemcpy(h->xq, p->xq, sizeof(double) * n * h->dq, cudaMemcpyDefault));
    CK(cudaMemcpy(h->y, p->y, sizeof(double) * n, cudaMemcpyDefault));
    {
        // column means of the training inputs (the centring of gpytorch's covar_dist, SURVEY A.3)
        std::vector<double> xh((size_t)n * std::max(h->dq, 1)), c(std::max(h->dq, 1), 0.0);
        if (h->dq > 0) CK(cudaMemcpy(xh.data(), p->xq, sizeof(double) * n * h->dq, cudaMemcpyDefault));
        for (int d = 0; d < h->dq; d++) {
            double sacc = 0.0;
            for (long long i = 0; i < n; i++) sacc += xh[i * h->dq + d];
            c[d] = sacc / (double)n;
        }
        CK(cudaMemcpy(h->centre, c.data(), sizeof(double) * std::max(h->dq, 1), cudaMemcpyHostToDevice));
    }
    auto upload_idx = [&](const int32_t* src, int* slot, int** dst, int hi, const char* name) -> int {
        *dst = nullptr;
        if (!src) return GPP_OK;
        std::vector<int> tmp((size_t)n);
        cudaError_t e = cudaMemcpy(tmp.data(), src, sizeof(int) * n, cudaMemcpyDefault);
        if (e != cudaSuccess) {
            set_err("index upload", e);
            return GPP_ERR_CUDA;
        }
        for (long long i = 0; i < n; i++)
            if (tmp[i] >= hi || tmp[i] < -1) {
                g_err = std::string("gpp_create: ") + name + " out of range";
                return GPP_ERR_ARG;
            }
        e = cudaMemcpy(slot, tmp.data(), sizeof(int) * n, cudaMemcpyHostToDevice);
        if (e != cudaSuccess) {
            set_err("index upload", e);
            return GPP_ERR_CUDA;
        }
        *dst = slot;
        if (dst == &h->level_idx) h->level_idx_host = tmp;
        return GPP_OK;
    };
    int rc;
    if (h->dz > 0 && (rc = upload_idx(p->level_idx, h->idx_slots[0], &h->level_idx, h->n_combo, "level_idx")) != GPP_OK)
        return rc;
    if ((rc = upload_idx(p->noise_idx, h->idx_slots[1], &h->noise_idx, h->n_noise, "noise_idx")) != GPP_OK) return rc;
    if ((rc = upload_idx(p->mean_idx, h->idx_slots[2], &h->mean_idx, std::max(h->n_mean, 1), "mean_idx")) != GPP_OK)
        return rc;
    return GPP_OK;
}

extern "C" int gpp_create(const gpp_problem* p, int device, gpp_handle** out) {
    if (!p || !out) ARG_FAIL("gpp_create: null argument");
    *out = nullptr;
    if (p->n <= 0 || p->n > (1 << 20)) ARG_FAIL("gpp_create: n out of range");
    if (p->dq < 0 || p->dq > GPP_MAX_DQ) ARG_FAIL("gpp_create: dq out of range");
    if (p->dz < 0 || p->dz > GPP_MAX_DZ) ARG_FAIL("gpp_create: dz out of range");
    if (p->dq == 0 && p->dz == 0) ARG_FAIL("gpp_create: no inputs");
    if (p->dz > 0 && (p->n_combo <= 0 || !p->level_idx)) ARG_FAIL("gpp_create: latent map needs n_combo and level_idx");
    if (p->n_noise < 1 || p->n_mean < 0) ARG_FAIL("gpp_create: n_noise must be >= 1 and n_mean >= 0");
    if (p->kernel < 0 || p->kernel > 2) ARG_FAIL("gpp_create: unknown kernel");
    if (p->n_pass < 0 || p->n_pass > 64) ARG_FAIL("gpp_create: n_pass out of range (0..64)");
    if (p->n_pass > 1 && p->dz == 0) ARG_FAIL("gpp_create: several latent passes need a latent map (dz > 0)");
    if ((p->dq > 0 && !p->xq) || !p->y) ARG_FAIL("gpp_create: xq / y missing");
    int ndev = gpp_device_count();
    if (ndev <= 0) {
        g_err = "gpp_create: no CUDA device visible (this engine has no CPU path)";
        return GPP_ERR_CUDA;
    }
    if (device < 0 || device >= ndev) ARG_FAIL("gpp_create: bad device index");
    CK(cudaSetDevice(device));
    // (cudaGetDeviceProperties costs milliseconds per call; the lock-step driver creates dozens of handles per fit)
    int cc_major = 0;
    CK(cudaDeviceGetAttribute(&cc_major, cudaDevAttrComputeCapabilityMajor, device));
    if (cc_major < 10) {
        g_err = "gpp_create: built for sm_100a (B200); device compute capability is too old";
        return GPP_ERR_CUDA;
    }

    const CreateConfig cfg = read_config((int)((p->n + 127) / 128));
    {
        // a parked handle of the same shape and configuration on this device: re-upload the data, keep everything else
        gpp_handle* reuse = nullptr;
        {
            std::lock_guard<std::mutex> lk(g_pool_mu);
            for (size_t i = 0; i < g_pool.size(); i++)
                if (same_shape(g_pool[i], p, device, cfg)) {
                    reuse = g_pool[i];
                    g_pool_bytes -= reuse->slab_bytes;
                    g_pool.erase(g_pool.begin() + (long)i);
                    break;
                }
        }
        if (reuse) {
            memset(&reuse->stats, 0, sizeof(reuse->stats));
            reuse->use_graph = cfg.graph != 0;   // (a failed graph capture may have switched the replay off)
            int rc = upload_problem(reuse, p);
            if (rc != GPP_OK) {
                destroy_now(reuse);
                return rc;
            }
            *out = reuse;
            return GPP_OK;
        }
    }

    gpp_handle* h = new gpp_handle();
    h->cfg = cfg;
    h->use_graph = cfg.graph != 0;
    memset(&h->tm, 0, sizeof(h->tm));
    memset(&h->stats, 0, sizeof(h->stats));
    for (int i = 0; i < EV_COUNT; i++) h->ev_valid[i] = false;
    h->device = device;
    h->n = p->n;
    h->np = (p->n + 127) / 128 * 128;
    h->T = (int)(h->np / 128);
    h->dq = p->dq;
    h->dqp = pad_dq(p->dq);
    h->dz = p->dz;
    h->n_combo = p->dz > 0 ? p->n_combo : 0;
    h->n_noise = p->n_noise;
    h->n_mean = p->n_mean;
    h->kernel = p->kernel;
    h->n_pass = p->n_pass > 1 ? p->n_pass : 1;
    const long long n = h->n, np = h->np;
    const int T = h->T;

#define CKH(x)                    \
    do {                          \
        cudaError_t e_ = (x);     \
        if (e_ != cudaSuccess) {  \
            set_err(#x, e_);      \
            destroy_now(h);       \
            return GPP_ERR_CUDA;  \
        }                         \
    } while (0)

    {
        // optional: sleep instead of spinning in cudaStreamSynchronize (many restart workers per GPU); must be
        // set before the context is created, so it only takes effect for the first handle of a process
        const char* e = getenv("GPP_BLOCKING_SYNC");
        if (e && atoi(e) != 0) {
            if (cudaSetDeviceFlags(cudaDeviceScheduleBlockingSync) != cudaSuccess) cudaGetLastError();
        }
    }
    {
        // three priority classes: panel chain (side stream, highest) > this stream > overlapped inverse (lowest)
        int lo = 0, hi = 0;
        CKH(cudaDeviceGetStreamPriorityRange(&lo, &hi));
        CKH(cudaStreamCreateWithPriority(&h->st, cudaStreamNonBlocking, (lo + hi) / 2));
    }
    for (int i = 0; i < EV_COUNT; i++) CKH(cudaEventCreate(&h->ev[i]));
    CKH(cudaEventCreateWithFlags(&h->ev_info, cudaEventDisableTiming));
    {
        // dynamic shared-memory limits of the kernels: once per device and process
        static std::mutex mu;
        static bool done[64] = {false};
        std::lock_guard<std::mutex> lk(mu);
        if (device >= 64 || !done[device]) {
            CKH(chol_set_attributes());
            CKH(cov_set_attributes());
            if (device < 64) done[device] = true;
        }
    }
    h->la.sched = cfg.chol;
    CKH(h->la.init(h->T));
    if (cfg.int8) {
        h->oz = new OzCtx();
        h->oz->sched = cfg.oz;
        cudaError_t oe = h->oz->init((int)h->np);
        if (oe == cudaErrorMemoryAllocation) {
            // the digit planes (3 x 7 Np^2 bytes) do not fit next to the FP64 work matrices: stay on DMMA
            cudaGetLastError();
            h->oz->destroy();
            delete h->oz;
            h->oz = nullptr;
        } else {
            CKH(oe);
        }
    }

    h->hyp_len = h->dq + h->n_pass * h->n_combo * h->dz + h->n_noise + h->n_mean + 2;
    h->res_len = 4 + h->dq + h->n_noise + h->n_mean;
    {
        // ONE device allocation and ONE pinned allocation per handle: the lock-step multi-start driver creates up to
        // 64 handles per fit, and ~45 separate cudaMalloc / cudaMallocHost calls per handle dominated its start-up
        size_t off = 0;
        auto take = [&](size_t bytes) {
            size_t at = off;
            off += (std::max<size_t>(bytes, 8) + 255) / 256 * 256;
            return at;
        };
        const size_t D = sizeof(double), I = sizeof(int);
        const size_t o_xq = take(D * n * h->dq), o_y = take(D * n), o_centre = take(D * std::max(h->dq, 1));
        const size_t o_lvl = take(I * n), o_nidx = take(I * n), o_midx = take(I * n);
        const size_t o_hyp = take(D * h->hyp_len), o_xs = take(D * np * h->dqp), o_xst = take(D * np * h->dqp), o_nrm = take(D * np);
        const size_t o_zpt = take(D * h->n_pass * np * ZP), o_r = take(D * np), o_da = take(D * np), o_v = take(D * np);
        const size_t o_alpha = take(D * np), o_part = take(D * T * np);
        const size_t o_A = take(D * np * np), o_M = take(D * np * np), o_S = take(D * np * np);
        const size_t o_ld = take(D * T), o_info = take(I);
        const size_t o_tp = take(D * h->n_pass * (size_t)T * (T + 1) / 2 * (1 + h->dqp));
        const size_t o_zpart = take(h->dz > 0 ? D * h->n_pass * T * np * ZP : 8);
        const size_t o_gz = take(h->dz > 0 ? D * h->n_pass * n * h->dz : 8);
        const size_t o_res = take(D * h->res_len);
        CKH(cudaMalloc(&h->slab, off));
        char* base = (char*)h->slab;
        h->xq = (double*)(base + o_xq);
        h->y = (double*)(base + o_y);
        h->centre = (double*)(base + o_centre);
        h->hyp = (double*)(base + o_hyp);
        h->xs = (double*)(base + o_xs);
        h->xst = (double*)(base + o_xst);
        h->nrm = (double*)(base + o_nrm);
        h->zpt = (double*)(base + o_zpt);
        h->r = (double*)(base + o_r);
        h->diag_add = (double*)(base + o_da);
        h->v = (double*)(base + o_v);
        h->alpha = (double*)(base + o_alpha);
        h->part = (double*)(base + o_part);
        h->A = (double*)(base + o_A);
        h->M = (double*)(base + o_M);
        h->S = (double*)(base + o_S);
        h->logdet_part = (double*)(base + o_ld);
        h->info = (int*)(base + o_info);
        h->tile_part = (double*)(base + o_tp);
        if (h->dz > 0) {
            h->zpart = (double*)(base + o_zpart);
            h->gz = (double*)(base + o_gz);
        }
        h->res = (double*)(base + o_res);
        h->idx_slots[0] = (int*)(base + o_lvl);
        h->idx_slots[1] = (int*)(base + o_nidx);
        h->idx_slots[2] = (int*)(base + o_midx);
        h->slab_bytes = off;

        size_t poff = 0;
        auto ptake = [&](size_t bytes) {
            size_t at = poff;
            poff += (std::max<size_t>(bytes, 8) + 63) / 64 * 64;
            return at;
        };
        const size_t p_hyp = ptake(D * h->hyp_len), p_info = ptake(I), p_res = ptake(D * h->res_len);
        const size_t p_gz = ptake(h->dz > 0 ? D * h->n_pass * n * h->dz : 8);
        CKH(cudaMallocHost(&h->pinned_slab, poff));
        char* pb = (char*)h->pinned_slab;
        h->hyp_host = (double*)(pb + p_hyp);
        h->info_host = (int*)(pb + p_info);
        h->res_host = (double*)(pb + p_res);
        if (h->dz > 0) h->gz_host = (double*)(pb + p_gz);
    }
    {
        int rc = upload_problem(h, p);
        if (rc != GPP_OK) {
            destroy_now(h);
            return rc;
        }
    }
    CKH(cudaMemsetAsync(h->M, 0, sizeof(double) * np * np, h->st));
    CKH(cudaStreamSynchronize(h->st));
#undef CKH
    *out = h;
    return GPP_OK;
}

static void mark(gpp_handle* h, int which) {
    if (h->capturing) return;  // timing events cannot live inside a captured graph
    cudaEventRecord(h->ev[which], h->st);
    h->ev_valid[which] = true;
}

static float span(gpp_handle* h, int a, int b) {
    if (!h->ev_valid[a] || !h->ev_valid[b]) return 0.f;
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, h->ev[a], h->ev[b]) != cudaSuccess) {
        cudaGetLastError();
        return 0.f;
    }
    return ms;
}

static int check_hyper(const gpp_handle* h, const gpp_hyper* hy) {
    if (!hy) ARG_FAIL("hyper: null");
    if (h->dq > 0 && !hy->w) ARG_FAIL("hyper: w missing");
    if (h->dz > 0 && !hy->z) ARG_FAIL("hyper: latent table z missing");
    if (!hy->noise) ARG_FAIL("hyper: noise missing");
    if (h->n_mean > 0 && !hy->beta) ARG_FAIL("hyper: beta missing");
    return GPP_OK;
}

// hyper-parameters of this evaluation into the pinned staging buffer
static void fill_hyper_host(gpp_handle* h, const gpp_hyper* hy, double jitter) {
    double* hh = h->hyp_host;
    int o = 0;
    for (int d = 0; d < h->dq; d++) hh[o++] = hy->w[d];
    for (int k = 0; k < ztab_len(h); k++) hh[o++] = hy->z[k];
    for (int k = 0; k < h->n_noise; k++) hh[o++] = hy->noise[k];
    for (int k = 0; k < h->n_mean; k++) hh[o++] = hy->beta[k];
    hh[o++] = hy->sigma_f2;
    hh[o++] = jitter;
    h->sf2 = hy->sigma_f2;
}

// point panels of n points (rows np, padding rows zero) from their inputs xq [n x dq] and latent levels (NULL without a
// latent map) with the current hyper-parameters; xst, the feature-major copy, may be NULL
static int prep_panels(gpp_handle* h, const double* xq, const int* level_idx, long long n, long long np, double* xs,
                       double* xst, double* nrm, double* zpt) {
    PrepArgs pa;
    pa.xq = xq;
    pa.level_idx = level_idx;
    pa.w = hyp_w(h);
    pa.centre = h->centre;
    pa.ztab = hyp_z(h);
    pa.n = (int)n;
    pa.np = (int)np;
    pa.dq = h->dq;
    pa.dqp = h->dqp;
    pa.dz = h->dz;
    pa.n_combo = h->n_combo;
    pa.n_pass = h->n_pass;
    pa.xs = xs;
    pa.xst = xst;
    pa.nrm = nrm;
    pa.zpt = zpt;
    prep_points_kernel<<<(int)((np + 255) / 256), 256, 0, h->st>>>(pa);
    CK(cudaGetLastError());
    count_launch();
    return GPP_OK;
}

// prepared panels of a set of points as rows or columns of a covariance block: n points in `tiles` 128-row tiles,
// xs [tiles*128 x dqp], nrm, and n_pass latent tables of zs doubles each from zpt
struct Panels {
    const double *xs, *nrm, *zpt;
    long long zs;
    int n, tiles;
};

static Panels training_panels(const gpp_handle* h) { return {h->xs, h->nrm, h->zpt, h->np * ZP, (int)h->n, h->T}; }

// covariance block of the rows r against the columns c, K = (1/n_pass) sum_p K_p: one launch per latent table.  `ca`
// carries the block's own options (out, ld, tri, same, pad_identity, sf2_dev, diag_add, alpha, mean_part, ld_part).
static int launch_cov_passes(const gpp_handle* h, CovArgs ca, const Panels& r, const Panels& c) {
    ca.xs_r = r.xs;
    ca.nrm_r = r.nrm;
    ca.n_r = r.n;
    ca.tiles_r = r.tiles;
    ca.xs_c = c.xs;
    ca.nrm_c = c.nrm;
    ca.n_c = c.n;
    ca.tiles_c = c.tiles;
    ca.dqp = h->dqp;
    ca.dz = h->dz;
    ca.sf2 = h->sf2;
    ca.scale = 1.0 / (double)h->n_pass;
    for (int p = 0; p < h->n_pass; p++) {
        ca.zpt_r = r.zpt + (size_t)p * r.zs;
        ca.zpt_c = c.zpt + (size_t)p * c.zs;
        ca.accum = p > 0;
        ca.last = p == h->n_pass - 1;
        CK(launch_cov(ca, h->kernel, h->st));
    }
    return GPP_OK;
}

// upload the staged hyper-parameters and prepare the per-point panels of the training set
static int stage_prep(gpp_handle* h) {
    CK(cudaMemcpyAsync(h->hyp, h->hyp_host, sizeof(double) * h->hyp_len, cudaMemcpyHostToDevice, h->st));
    int rc = prep_panels(h, h->xq, h->level_idx, h->n, h->np, h->xs, h->xst, h->nrm, h->zpt);
    if (rc != GPP_OK) return rc;
    const int nb = (int)((h->np + 255) / 256);
    prep_targets_kernel<<<nb, 256, 0, h->st>>>(h->y, h->mean_idx, hyp_beta(h), h->n_mean, h->noise_idx, hyp_noise(h),
                                                h->n_noise, 0.0, hyp_jitter(h), (int)h->n, (int)h->np, h->r,
                                                h->diag_add);
    CK(cudaGetLastError());
    count_launch();
    return GPP_OK;
}

// K_y (lower tiles) into A, then A -> L in place, diagonal blocks of M <- L_kk^-1 (status in h->info)
static int stage_factor(gpp_handle* h) {
    CK(cudaMemsetAsync(h->info, 0, sizeof(int), h->st));
    CovArgs ca;
    memset(&ca, 0, sizeof(ca));
    ca.out = h->A;
    ca.ld = h->np;
    ca.tri = 1;
    ca.same = 1;
    ca.pad_identity = 1;
    ca.sf2_dev = hyp_sf2(h);
    ca.diag_add = h->diag_add;
    int rc = launch_cov_passes(h, ca, training_panels(h), training_panels(h));
    if (rc != GPP_OK) return rc;
    mark(h, EV_COV);
    if (h->cfg.small_block > 0 && h->T <= 16) {
        // small problems: the whole factorisation is one dataflow launch (block_potrf_kernel) instead of a chain of
        // T leaf / TRSM / update launches.  Inside a captured graph the launch arguments are frozen, so the tile flags
        // are cleared by a memset node and the epoch is constant.
        CK(cudaMemsetAsync(h->la.blk_flags, 0, 256 * sizeof(int), h->st));
        CK(launch_block_potrf(h->A, h->M, (int)h->np, 0, h->T, h->logdet_part, h->info, h->la.blk_flags, 1,
                              h->cfg.small_block, h->st));
    } else if (h->cfg.lookahead && h->oz && h->oz->ready && h->T >= h->oz->sched.lazy_min_tiles)
        CK(potrf_lazy(h->A, h->M, (int)h->np, h->T, h->logdet_part, h->info, h->st, h->la, h->S, *h->oz));
    else if (h->cfg.lookahead)
        CK(potrf_lookahead(h->A, h->M, (int)h->np, h->T, h->logdet_part, h->info, h->st, h->la, h->S, h->oz));
    else
        CK(potrf_blocked(h->A, h->M, (int)h->np, h->T, h->logdet_part, h->info, h->st));
    mark(h, EV_CHOL);
    return GPP_OK;
}

// M <- L^-1, v = M r, alpha = M^T v
static int stage_inverse_solve(gpp_handle* h) {
    if (h->cfg.lookahead && h->la.inv_pending) {
        // the leading part of L^-1 was started behind the factorisation (trtri_early): join it, finish the rest
        CK(cudaStreamWaitEvent(h->st, h->la.inv_done, 0));
        h->la.inv_pending = false;
        CK(trtri_late(h->A, h->M, h->S, (int)h->np, h->T, h->st, h->oz));
    } else {
        CK(trtri_doubling(h->A, h->M, h->S, (int)h->np, h->T, h->st, h->oz));
    }
    mark(h, EV_TRTRI);
    trmv_lower_kernel<<<(int)(h->np / 8), 256, 0, h->st>>>(h->M, h->np, h->r, (int)h->np, h->v);
    CK(cudaGetLastError());
    count_launch();
    trmv_lower_t_part_kernel<<<h->T * (h->T + 1) / 2, 512, 0, h->st>>>(h->M, h->np, h->v, (int)h->np, h->part);
    CK(cudaGetLastError());
    count_launch();
    trmv_lower_t_reduce_kernel<<<(int)((h->np + 255) / 256), 256, 0, h->st>>>(h->part, (int)h->np, h->T, h->alpha);
    CK(cudaGetLastError());
    count_launch();
    mark(h, EV_SOLVE);
    return GPP_OK;
}

static int stage_grad(gpp_handle* h) {
    CK(lauum_full(h->M, h->S, (int)h->np, h->T, h->st, 0, h->oz));
    mark(h, EV_LAUUM);
    GradArgs ga;
    memset(&ga, 0, sizeof(ga));
    ga.xst = h->xst;
    ga.nrm = h->nrm;
    ga.alpha = h->alpha;
    ga.Kinv = h->S;
    ga.ld = h->np;
    ga.n = (int)h->n;
    ga.np = (int)h->np;
    ga.T = h->T;
    ga.dq = h->dq;
    ga.dqp = h->dqp;
    ga.dz = h->dz;
    ga.sf2 = h->sf2;
    ga.sf2_dev = hyp_sf2(h);
    const size_t tp_stride = (size_t)h->T * (h->T + 1) / 2 * (1 + h->dqp);
    const size_t zp_stride = (size_t)h->T * h->np * ZP;
    // every gradient component is linear in K, so the gradient of the averaged covariance is the average of the
    // single-table gradients evaluated with the SAME W = alpha alpha^T - K_y^-1: one pass per latent table
    for (int p = 0; p < h->n_pass; p++) {
        ga.zpt = h->zpt + (size_t)p * h->np * ZP;
        ga.tile_part = h->tile_part + p * tp_stride;
        ga.zpart = h->dz > 0 ? h->zpart + p * zp_stride : nullptr;
        CK(launch_grad(ga, h->kernel, h->st));
        if (h->dz > 0) {
            const int cnt = (int)(h->n * h->dz);
            zpart_reduce_kernel<<<(cnt + 255) / 256, 256, 0, h->st>>>(ga.zpart, h->T, (int)h->np, (int)h->n, h->dz,
                                                                      h->gz + (size_t)p * cnt, 1.0 / (double)h->n_pass);
            CK(cudaGetLastError());
            count_launch();
        }
    }
    if (h->dz > 0)
        CK(cudaMemcpyAsync(h->gz_host, h->gz, sizeof(double) * h->n_pass * h->n * h->dz, cudaMemcpyDeviceToHost,
                           h->st));
    mark(h, EV_GRAD);
    return GPP_OK;
}

static int stage_finish(gpp_handle* h, int want_grad) {
    FinishArgs fa;
    memset(&fa, 0, sizeof(fa));
    fa.v = h->v;
    fa.alpha = h->alpha;
    fa.logdet_part = h->logdet_part;
    fa.Kinv = h->S;
    fa.ld = h->np;
    fa.tile_part = h->tile_part;
    fa.w = hyp_w(h);
    fa.noise_idx = h->noise_idx;
    fa.mean_idx = h->mean_idx;
    fa.info = h->info;
    fa.n = (int)h->n;
    fa.np = (int)h->np;
    fa.T = h->T;
    fa.dq = h->dq;
    fa.dqp = h->dqp;
    fa.n_noise = h->n_noise;
    fa.n_mean = h->n_mean;
    fa.want_grad = want_grad;
    fa.n_pass = h->n_pass;
    fa.res = h->res;
    finish_kernel<<<1, 256, 0, h->st>>>(fa);
    CK(cudaGetLastError());
    count_launch();
    CK(cudaMemcpyAsync(h->res_host, h->res, sizeof(double) * h->res_len, cudaMemcpyDeviceToHost, h->st));
    return GPP_OK;
}

static const double kJitter[4] = {0.0, 1e-8, 1e-7, 1e-6};  // psd_safe_cholesky ladder (SURVEY A.5)

// every device operation of one evaluation, in stream order, without host synchronisation
static int enqueue_eval(gpp_handle* h, int want_grad) {
    int rc;
    if ((rc = stage_prep(h)) != GPP_OK) return rc;
    if ((rc = stage_factor(h)) != GPP_OK) return rc;
    if ((rc = stage_inverse_solve(h)) != GPP_OK) return rc;
    if (want_grad && (rc = stage_grad(h)) != GPP_OK) return rc;
    return stage_finish(h, want_grad);
}

// capture enqueue_eval once per (handle, want_grad); returns false when capture is not possible
static bool ensure_graph(gpp_handle* h, int want_grad) {
    const int slot = want_grad ? 1 : 0;
    if (h->graph_exec[slot]) return true;
    if (cudaStreamBeginCapture(h->st, cudaStreamCaptureModeThreadLocal) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    const long long k0 = t_launches;
    h->capturing = true;
    const int rc = enqueue_eval(h, want_grad);
    h->capturing = false;
    cudaGraph_t g = nullptr;
    cudaError_t e = cudaStreamEndCapture(h->st, &g);
    const long long kernels = t_launches - k0;  // launches issued by THIS thread while capturing
    g_launches.fetch_sub(kernels);              // captured, not executed
    if (rc != GPP_OK || e != cudaSuccess || !g) {
        if (g) cudaGraphDestroy(g);
        cudaGetLastError();
        return false;
    }
    cudaGraphExec_t ex = nullptr;
    e = cudaGraphInstantiate(&ex, g, 0);
    cudaGraphDestroy(g);
    if (e != cudaSuccess || !ex) {
        cudaGetLastError();
        return false;
    }
    h->graph_exec[slot] = ex;
    h->graph_kernels[slot] = kernels;
    return true;
}

// large problems (no graph replay): the factorisation status is read back as soon as the factorisation is done, so
// that a failed rung of the jitter ladder costs the covariance build + factorisation only (about 40 % of an
// evaluation with gradient) instead of the inverse, K^-1 and the gradient pass on top of a garbage factor
static int enqueue_eval_early_out(gpp_handle* h, int want_grad, int* failed) {
    int rc;
    *failed = 0;
    if ((rc = stage_prep(h)) != GPP_OK) return rc;
    if ((rc = stage_factor(h)) != GPP_OK) return rc;
    CK(cudaMemcpyAsync(h->info_host, h->info, sizeof(int), cudaMemcpyDeviceToHost, h->st));
    CK(cudaEventRecord(h->ev_info, h->st));
    CK(cudaEventSynchronize(h->ev_info));
    if (*h->info_host != 0) {
        *failed = *h->info_host;
        if (h->cfg.lookahead && h->la.inv_pending) {
            // the leading part of L^-1 was started behind the factorisation: let it drain before A / M are reused
            CK(cudaStreamWaitEvent(h->st, h->la.inv_done, 0));
            h->la.inv_pending = false;
        }
        h->stats.early_outs++;
        return GPP_OK;
    }
    if ((rc = stage_inverse_solve(h)) != GPP_OK) return rc;
    if (want_grad && (rc = stage_grad(h)) != GPP_OK) return rc;
    return stage_finish(h, want_grad);
}

// one evaluation with the jitter ladder; on success L is in A, L^-1 in M, alpha / res_host are valid
static int run_eval(gpp_handle* h, const gpp_hyper* hy, int want_grad, int first_rung = 0) {
    if (first_rung == 0) h->stats.evaluations++;
    for (int a = first_rung; a < 4; a++) {
        for (int i = 0; i < EV_COUNT; i++) h->ev_valid[i] = false;
        fill_hyper_host(h, hy, kJitter[a]);
        if (h->use_graph && !ensure_graph(h, want_grad)) h->use_graph = false;
        h->stats.factorizations++;
        if (a > 0) h->stats.jitter_retries++;
        mark(h, EV_START);
        int info;
        if (h->use_graph) {
            CK(cudaGraphLaunch(h->graph_exec[want_grad ? 1 : 0], h->st));
            count_launch((int)h->graph_kernels[want_grad ? 1 : 0]);
            mark(h, EV_END);
            CK(cudaStreamSynchronize(h->st));
            info = (int)h->res_host[2];
        } else {
            int failed = 0;
            int rc = enqueue_eval_early_out(h, want_grad, &failed);
            if (rc != GPP_OK) return rc;
            mark(h, EV_END);
            CK(cudaStreamSynchronize(h->st));
            if (h->la.sched.timeline)
                h->la.dump_timeline(h->oz ? (h->T + h->oz->sched.lazy_pb - 1) / h->oz->sched.lazy_pb : h->la.panels);
            info = failed ? failed : (int)h->res_host[2];
        }
        if (info & 2) {
            g_err = "NaN encountered while factorising K_y";
            return GPP_ERR_NAN;
        }
        if (info == 0) {
            h->last_jitter = kJitter[a];
            return GPP_OK;
        }
    }
    g_err = "K_y not positive definite after adding jitter up to 1e-6";
    return GPP_ERR_NOT_PD;
}

// results of the evaluation that just completed on h->st (res_host / gz_host are valid) into `out`
static int collect_mll(gpp_handle* h, int want_grad, gpp_mll_result* out) {
    const double* r = h->res_host;
    out->quad = r[0];
    out->logdet = r[1];
    out->jitter = h->last_jitter;
    out->nll = 0.5 * (r[0] + r[1] + (double)h->n * 1.8378770664093453);
    if (!(out->nll == out->nll)) {
        g_err = "NaN in the marginal likelihood";
        return GPP_ERR_NAN;
    }
    if (want_grad) {
        out->d_sigma_f2 = r[3];
        if (out->d_w)
            for (int d = 0; d < h->dq; d++) out->d_w[d] = r[4 + d];
        if (out->d_noise)
            for (int k = 0; k < h->n_noise; k++) out->d_noise[k] = r[4 + h->dq + k];
        if (out->d_beta)
            for (int k = 0; k < h->n_mean; k++) out->d_beta[k] = r[4 + h->dq + h->n_noise + k];
        if (out->d_z && h->dz > 0) {
            // d nll / d Z[a] = sum_{i in a} sum_j P_ij (z_i - z_j): scatter the per-point sums by level
            for (int k = 0; k < ztab_len(h); k++) out->d_z[k] = 0.0;
            for (int p = 0; p < h->n_pass; p++) {
                double* dz_p = out->d_z + (size_t)p * h->n_combo * h->dz;
                const double* gz_p = h->gz_host + (size_t)p * h->n * h->dz;
                for (long long i = 0; i < h->n; i++) {
                    int a = h->level_idx_host[(size_t)i];
                    if (a < 0) continue;
                    for (int k = 0; k < h->dz; k++) dz_p[a * h->dz + k] += gz_p[i * h->dz + k];
                }
            }
        }
    } else {
        out->d_sigma_f2 = 0.0;
    }
    h->tm.covariance = span(h, EV_START, EV_COV);
    h->tm.cholesky = span(h, EV_COV, EV_CHOL);
    h->tm.trtri = span(h, EV_CHOL, EV_TRTRI);
    h->tm.solve = span(h, EV_TRTRI, EV_SOLVE);
    h->tm.lauum = want_grad ? span(h, EV_SOLVE, EV_LAUUM) : 0.f;
    h->tm.gradient = want_grad ? span(h, EV_LAUUM, EV_GRAD) : 0.f;
    h->tm.total = span(h, EV_START, EV_END);
    return GPP_OK;
}

extern "C" int gpp_mll_grad(gpp_handle* h, const gpp_hyper* hy, int want_grad, gpp_mll_result* out) {
    if (!h || !out) ARG_FAIL("gpp_mll_grad: null argument");
    int rc = check_hyper(h, hy);
    if (rc != GPP_OK) return rc;
    CK(cudaSetDevice(h->device));
    h->factorized = false;
    h->fgen++;
    h->pending = false;
    rc = run_eval(h, hy, want_grad ? 1 : 0);
    if (rc != GPP_OK) return rc;
    h->factorized = true;
    h->fgen++;
    return collect_mll(h, want_grad, out);
}

extern "C" int gpp_set_theta_layout(gpp_handle* h, const gpp_theta_layout* layout) {
    if (!h || !layout) ARG_FAIL("gpp_set_theta_layout: null argument");
    if (h->n_pass > 1) ARG_FAIL("gpp_set_theta_layout: the closed-form layout covers the single-pass latent map only");
    const char* err = layout_copy(h->layout, layout, h->dq, h->dz, h->n_combo, h->n_noise, h->n_mean);
    if (err) {
        h->layout.set = false;
        ARG_FAIL(err);
    }
    h->g_w.assign(std::max(h->dq, 1), 0.0);
    h->g_z.assign(std::max(h->n_pass * h->n_combo * h->dz, 1), 0.0);
    h->g_noise.assign(std::max(h->n_noise, 1), 0.0);
    h->g_beta.assign(std::max(h->n_mean, 1), 0.0);
    return GPP_OK;
}

static gpp_hyper layout_hyper(gpp_handle* h) {
    ThetaLayout& L = h->layout;
    gpp_hyper hy;
    hy.w = L.w.data();
    hy.z = h->dz > 0 ? L.z.data() : nullptr;
    hy.sigma_f2 = L.sf2;
    hy.noise = L.noise.data();
    hy.beta = h->n_mean > 0 ? L.beta.data() : nullptr;
    return hy;
}

// chain rule to the raw parameters + log-priors on top of a finished evaluation
static int finish_objective(gpp_handle* h, int want_grad, double* value, double* grad, gpp_mll_result* detail) {
    ThetaLayout& L = h->layout;
    gpp_mll_result r;
    memset(&r, 0, sizeof(r));
    r.d_w = h->g_w.data();
    r.d_z = h->g_z.data();
    r.d_noise = h->g_noise.data();
    r.d_beta = h->g_beta.data();
    int rc = collect_mll(h, want_grad, &r);
    if (rc != GPP_OK) return rc;
    if (want_grad) layout_chain(L, r, h->dq, h->dz, h->n_combo, h->n_noise, h->n_mean, grad);
    const double logp = layout_priors(L, want_grad ? grad : nullptr);
    *value = r.nll - logp;
    if (detail) {
        detail->nll = r.nll;
        detail->logdet = r.logdet;
        detail->quad = r.quad;
        detail->jitter = r.jitter;
        detail->d_sigma_f2 = r.d_sigma_f2;
    }
    if (!(*value == *value)) {
        g_err = "NaN in the objective";
        return GPP_ERR_NAN;
    }
    return GPP_OK;
}

extern "C" int gpp_objective(gpp_handle* h, const double* theta, int want_grad, double* value, double* grad,
                             gpp_mll_result* detail) {
    if (!h || !theta || !value) ARG_FAIL("gpp_objective: null argument");
    if (!h->layout.set) ARG_FAIL("gpp_objective: call gpp_set_theta_layout first");
    if (want_grad && !grad) ARG_FAIL("gpp_objective: grad missing");
    layout_natural(h->layout, theta, h->dq, h->dz, h->n_combo, h->n_noise, h->n_mean);
    gpp_hyper hy = layout_hyper(h);
    CK(cudaSetDevice(h->device));
    h->factorized = false;
    h->fgen++;
    h->pending = false;
    int rc = run_eval(h, &hy, want_grad ? 1 : 0);
    if (rc != GPP_OK) return rc;
    h->factorized = true;
    h->fgen++;
    return finish_objective(h, want_grad, value, grad, detail);
}

// Split form of gpp_objective for callers that keep MANY handles in flight from one host thread (the lock-step
// multi-start driver of fit_model_scipy): enqueue issues the whole evaluation on the handle's stream and returns
// without waiting; collect waits for it, walks the rest of the jitter ladder if the first factorisation failed, and
// applies the chain rule and the priors.  Values are identical to gpp_objective.
extern "C" int gpp_objective_enqueue(gpp_handle* h, const double* theta, int want_grad) {
    if (!h || !theta) ARG_FAIL("gpp_objective_enqueue: null argument");
    if (!h->layout.set) ARG_FAIL("gpp_objective_enqueue: call gpp_set_theta_layout first");
    if (h->pending) ARG_FAIL("gpp_objective_enqueue: the previous evaluation has not been collected");
    layout_natural(h->layout, theta, h->dq, h->dz, h->n_combo, h->n_noise, h->n_mean);
    gpp_hyper hy = layout_hyper(h);
    CK(cudaSetDevice(h->device));
    h->factorized = false;
    h->fgen++;
    h->stats.evaluations++;
    h->stats.factorizations++;
    const int wg = want_grad ? 1 : 0;
    for (int i = 0; i < EV_COUNT; i++) h->ev_valid[i] = false;
    fill_hyper_host(h, &hy, kJitter[0]);
    if (h->use_graph && !ensure_graph(h, wg)) h->use_graph = false;
    if (h->use_graph) {
        CK(cudaGraphLaunch(h->graph_exec[wg], h->st));
        count_launch((int)h->graph_kernels[wg]);
    } else {
        int rc = enqueue_eval(h, wg);
        if (rc != GPP_OK) return rc;
    }
    h->pending = true;
    h->pending_grad = wg;
    return GPP_OK;
}

extern "C" int gpp_objective_collect(gpp_handle* h, double* value, double* grad, gpp_mll_result* detail) {
    if (!h || !value) ARG_FAIL("gpp_objective_collect: null argument");
    if (!h->pending) ARG_FAIL("gpp_objective_collect: nothing was enqueued");
    const int wg = h->pending_grad;
    if (wg && !grad) ARG_FAIL("gpp_objective_collect: grad missing");
    CK(cudaSetDevice(h->device));
    h->pending = false;
    CK(cudaStreamSynchronize(h->st));
    const int info = (int)h->res_host[2];
    if (info & 2) {
        g_err = "NaN encountered while factorising K_y";
        return GPP_ERR_NAN;
    }
    if (info != 0) {
        gpp_hyper hy = layout_hyper(h);  // the natural parameters of the enqueued theta are still in the layout
        int rc = run_eval(h, &hy, wg, 1);
        if (rc != GPP_OK) return rc;
    } else {
        h->last_jitter = kJitter[0];
    }
    h->factorized = true;
    h->fgen++;
    return finish_objective(h, wg, value, grad, detail);
}

extern "C" int gpp_get_timings(gpp_handle* h, gpp_timings* out) {
    if (!h || !out) ARG_FAIL("gpp_get_timings: null argument");
    *out = h->tm;
    return GPP_OK;
}

extern "C" int gpp_get_stats(gpp_handle* h, gpp_stats* out) {
    if (!h || !out) ARG_FAIL("gpp_get_stats: null argument");
    *out = h->stats;
    return GPP_OK;
}

extern "C" int gpp_covariance(gpp_handle* h, const gpp_hyper* hy, double* k_out) {
    if (!h || !k_out) ARG_FAIL("gpp_covariance: null argument");
    int rc = check_hyper(h, hy);
    if (rc != GPP_OK) return rc;
    CK(cudaSetDevice(h->device));
    h->factorized = false;
    h->fgen++;
    fill_hyper_host(h, hy, 0.0);
    if ((rc = stage_prep(h)) != GPP_OK) return rc;
    CovArgs ca;
    memset(&ca, 0, sizeof(ca));
    ca.out = h->S;
    ca.ld = h->np;
    ca.same = 1;
    if ((rc = launch_cov_passes(h, ca, training_panels(h), training_panels(h))) != GPP_OK) return rc;
    CK(cudaMemcpy2DAsync(k_out, sizeof(double) * h->n, h->S, sizeof(double) * h->np, sizeof(double) * h->n, h->n,
                         cudaMemcpyDefault, h->st));
    CK(cudaStreamSynchronize(h->st));
    return GPP_OK;
}

extern "C" int gpp_fetch(gpp_handle* h, int which, double* out) {
    if (!h || !out) ARG_FAIL("gpp_fetch: null argument");
    CK(cudaSetDevice(h->device));
    if (which == 3) {
        CK(cudaMemcpyAsync(out, h->alpha, sizeof(double) * h->n, cudaMemcpyDefault, h->st));
        CK(cudaStreamSynchronize(h->st));
        return GPP_OK;
    }
    if (which == 4) {
        // diag(K_y^-1): a strided copy of n doubles (loocv_rrmse, optim/mll_noise_continuation.py:28-42)
        CK(cudaMemcpy2DAsync(out, sizeof(double), h->S, sizeof(double) * (h->np + 1), sizeof(double), h->n,
                             cudaMemcpyDefault, h->st));
        CK(cudaStreamSynchronize(h->st));
        return GPP_OK;
    }
    const double* src = which == 0 ? h->A : (which == 1 ? h->M : (which == 2 ? h->S : nullptr));
    if (!src) ARG_FAIL("gpp_fetch: which must be 0..4");
    std::vector<double> tmp((size_t)h->n * h->n);
    CK(cudaMemcpy2DAsync(tmp.data(), sizeof(double) * h->n, src, sizeof(double) * h->np, sizeof(double) * h->n, h->n,
                         cudaMemcpyDeviceToHost, h->st));
    CK(cudaStreamSynchronize(h->st));
    if (which < 2)
        for (long long i = 0; i < h->n; i++)
            for (long long j = i + 1; j < h->n; j++) tmp[(size_t)(i * h->n + j)] = 0.0;
    else  // K_y^-1 is kept as its lower triangle on the device (the gradient pass reads lower tiles only)
        for (long long i = 0; i < h->n; i++)
            for (long long j = i + 1; j < h->n; j++) tmp[(size_t)(i * h->n + j)] = tmp[(size_t)(j * h->n + i)];
    CK(cudaMemcpy(out, tmp.data(), sizeof(double) * h->n * h->n, cudaMemcpyDefault));
    return GPP_OK;
}

extern "C" int gpp_factorize(gpp_handle* h, const gpp_hyper* hy) {
    if (!h) ARG_FAIL("gpp_factorize: null handle");
    int rc = check_hyper(h, hy);
    if (rc != GPP_OK) return rc;
    CK(cudaSetDevice(h->device));
    h->factorized = false;
    h->fgen++;
    rc = run_eval(h, hy, 0);
    if (rc != GPP_OK) return rc;
    h->factorized = true;
    h->fgen++;
    return GPP_OK;
}

// ---------------------------------------------------------------------------------------------
// Prediction.  Candidate rows reach mean and variance through the chunk front (K* against the training set, U = K* L^-T,
// predict_finish_kernel) in chunks of at most mc_alloc rows.  Three caller families each run their own chunk loop and
// add their own stages:
//   pointwise  gpp_predict, gpp_predict_grad, gpp_acq_argmax (predict_rows)
//   point set  J1 of gpp_predict_joint / gpp_sample_posterior, gpp_ipv_points (load_point_set)
//   t-batch    gpp_posterior_qbatch[_grad], gpp_acq_qbatch, gpp_nipv_qbatch (qbatch_front and the qbatch_* stages)
static long long round128(long long x) { return (x + 127) / 128 * 128; }

// a call's candidate rows as the caller passed them (host or device; noise_idx and mean_idx may be NULL) and the noise
// setting and floor of their predictive variance
struct Rows {
    const double* xq;
    const int32_t *level_idx, *noise_idx, *mean_idx;
    int include_noise;
    double min_var;
};

// The argument checks of every entry point that takes candidate rows, in the order they fire: `bad_count` is the entry
// point's message for a count outside its range, or NULL; xq and level_idx are needed when there are rows.
static int check_rows(const gpp_handle* h, const char* name, const char* bad_count, long long rows, const double* xq,
                      const int32_t* level_idx) {
    const char* why = nullptr;
    if (!h) why = "null handle";
    else if (!h->factorized) why = "call gpp_factorize (or gpp_mll_grad) first";
    else if (bad_count) why = bad_count;
    else if (h->dq > GPP_MAX_DQ) why = "at most GPP_MAX_DQ quantitative inputs";
    else if (rows > 0 && h->dq > 0 && !xq) why = "xq missing";
    else if (rows > 0 && h->dz > 0 && !level_idx) why = "level_idx missing";
    if (!why) return GPP_OK;
    g_err = std::string(name) + ": " + why;
    return GPP_ERR_ARG;
}

// chunk buffers of mc_alloc rows, their leading dimension: it only grows, and a K* chunk holds at most 2^27 doubles
// (1 GiB)
static int ensure_chunk_buffers(gpp_handle* h, long long m) {
    const long long cap = std::max(((1LL << 27) / h->np) / 128 * 128, 128LL);
    const long long mc = std::max(h->mc_alloc, std::min(round128(m), cap));
    cudaStream_t st = h->st;
    CK(h->c_xq.reserve(mc * std::max(h->dq, 1), st));
    CK(h->c_xs.reserve(mc * h->dqp, st));
    CK(h->c_nrm.reserve(mc, st));
    CK(h->c_zpt.reserve(mc * ZP * h->n_pass, st));
    CK(h->c_K.reserve(mc * h->np, st));
    CK(h->c_lvl.reserve(mc, st));
    CK(h->c_noise.reserve(mc, st));
    CK(h->c_mean.reserve(mc, st));
    CK(h->c_cost.reserve(mc, st));
    CK(h->c_mean_part.reserve(mc * h->T, st));
    CK(h->c_rowsq.reserve(mc * h->T, st));
    CK(h->c_mu.reserve(mc, st));
    CK(h->c_var.reserve(mc, st));
    CK(h->c_score.reserve(mc, st));
    CK(h->c_blk_best.reserve(mc / 256 + 1, st));
    CK(h->c_blk_idx.reserve(mc / 256 + 1, st));
    h->mc_alloc = mc;
    return GPP_OK;
}

// U = K* L^-T of one chunk, the per-column-tile gradient partials and the chunk's gradients (gradient and t-batch
// paths).  The partials take T*dq doubles per candidate each, so these paths cap their chunk at 2^24 / (T*dq)
// candidates (128 MiB per partial buffer; 4096 candidates at N = 16384, dq = 32); mean and variance do not depend on
// the chunking.
static int ensure_grad_buffers(gpp_handle* h) {
    long long step = ((1LL << 24) / ((long long)h->T * std::max(h->dq, 1))) / 128 * 128;
    step = std::min(std::max(step, 128LL), h->mc_alloc);
    CK(h->g_U.reserve(step * h->np, h->st));
    CK(h->g_part_m.reserve(step * h->T * h->dq, h->st));
    CK(h->g_part_v.reserve(step * h->T * h->dq, h->st));
    CK(h->g_dmean.reserve(step * h->dq, h->st));
    CK(h->g_dvar.reserve(step * h->dq, h->st));
    h->g_step = step;
    return GPP_OK;
}

// prepared panels of the chunk buffers' first mc rows
static Panels chunk_panels(const gpp_handle* h, long long mc) {
    const long long mcp = round128(mc);
    return {h->c_xs, h->c_nrm, h->c_zpt, mcp * ZP, (int)mc, (int)(mcp / CT)};
}

struct AcqSpec {
    const int32_t* cost_idx = nullptr;
    int n_cost = 0;
    const double* cost = nullptr;
    const int32_t* kind_by_cost = nullptr;
    const double* best_f = nullptr;
    int maximize = 1;
    double si = 0.0, y_min = 0.0, y_std = 1.0;
    double* scores = nullptr;
    double best_score = -INFINITY;
    long long best_index = -1;
};

// The chunk front: rows [base, base + mc) of the call, their inputs and groups in the chunk buffers, to mean and
// variance in c_mu / c_var.  `given` holds the rows' prepared panels (a point set), or is NULL: the panels are prepared
// into c_xs / c_nrm / c_zpt here.  U = K* L^-T goes to U (ld Np) when given, else only its row sums of squares are kept
// (bitwise the same either way).  `acq` adds the gpp_acq_argmax scores and per-block best.
static int chunk_front(gpp_handle* h, const Rows& r, long long base, long long mc, const Panels* given, double* U,
                       const AcqSpec* acq) {
    const long long MC = h->mc_alloc;
    const Panels rows = given ? *given : chunk_panels(h, mc);
    int rc;
    if (!given && (rc = prep_panels(h, h->c_xq, h->dz > 0 ? h->c_lvl.p : nullptr, mc, round128(mc), h->c_xs, nullptr,
                                    h->c_nrm, h->c_zpt)) != GPP_OK)
        return rc;
    CovArgs ca;
    memset(&ca, 0, sizeof(ca));
    ca.out = h->c_K;
    ca.ld = h->np;
    ca.alpha = h->alpha;
    ca.mean_part = h->c_mean_part;
    ca.ld_part = MC;
    if ((rc = launch_cov_passes(h, ca, rows, training_panels(h))) != GPP_OK) return rc;

    GemmOp op = gemm_default();  // U = K* L^-T: its row sums of squares, and U itself when asked
    op.A = h->c_K;
    op.lda = (int)h->np;
    op.B = h->M;
    op.ldb = (int)h->np;
    op.C = U;
    op.ldc = U ? (int)h->np : 0;
    op.tiles_m = op.tiles_m_last = rows.tiles;
    op.tiles_n = h->T;
    op.klo_c = 0;
    op.khi_sel = KSEL_TJ;
    op.khi_c = 1;
    op.epilogue = U ? EPI_STORE_ROWSQ : EPI_ROWSQ;
    op.rowsq = h->c_rowsq;
    op.rowsq_ld = (int)MC;
    CK(launch_gemm(op, true, true, 1, h->st));

    PredFinishArgs fa;
    memset(&fa, 0, sizeof(fa));
    fa.mean_part = h->c_mean_part;
    fa.rowsq = h->c_rowsq;
    fa.ldp = MC;
    fa.tiles_c = h->T;
    fa.m = (int)mc;
    fa.base = base;
    fa.sf2 = h->sf2;
    fa.mean_idx = r.mean_idx ? h->c_mean.p : nullptr;
    fa.beta = hyp_beta(h);
    fa.n_mean = h->n_mean;
    fa.noise_idx = r.noise_idx ? h->c_noise.p : nullptr;
    fa.noise = hyp_noise(h);
    fa.n_noise = h->n_noise;
    fa.include_noise = r.include_noise;
    fa.min_var = r.min_var;
    fa.mean_out = h->c_mu;
    fa.var_out = h->c_var;
    if (acq) {
        fa.cost_idx = acq->cost_idx ? h->c_cost.p : nullptr;
        fa.cost = h->acq_par;
        fa.best_f = h->acq_par + acq->n_cost;
        fa.kind_by_cost = h->acq_kind;
        fa.n_cost = acq->n_cost;
        fa.maximize = acq->maximize;
        fa.si = acq->si;
        fa.y_min = acq->y_min;
        fa.y_std = acq->y_std;
        fa.score_out = acq->scores ? h->c_score.p : nullptr;
        fa.blk_best = h->c_blk_best;
        fa.blk_idx = h->c_blk_idx;
    }
    predict_finish_kernel<<<(int)((mc + 255) / 256), 256, 0, h->st>>>(fa);
    CK(cudaGetLastError());
    count_launch();
    return GPP_OK;
}

// V = U L^-1 = K* K_y^-1 of `tiles` row tiles, U [rows x Np] -> V [rows x Np]: B(tj, k) = L^-1[k, tj], k in [tj, T)
static int v_gemm(gpp_handle* h, const double* U, double* V, int tiles) {
    GemmOp vo = gemm_default();
    vo.A = U;
    vo.lda = (int)h->np;
    vo.B = h->M;
    vo.ldb = (int)h->np;
    vo.C = V;
    vo.ldc = (int)h->np;
    vo.tiles_m = vo.tiles_m_last = tiles;
    vo.tiles_n = h->T;
    vo.klo_sel = KSEL_TJ;
    vo.klo_c = 0;
    vo.khi_c = h->T;
    CK(launch_gemm(vo, true, false, 1, h->st));
    return GPP_OK;
}

// predict_grad_tile_kernel partials [c.tiles * dq][ldp] of the rows r against the column points c: alpha weighs the
// mean partials, V [rows x ldv] the variance partials
static int grad_tiles(gpp_handle* h, const Panels& r, const Panels& c, const double* alpha, const double* V,
                      long long ldv, double* part_m, double* part_v, long long ldp) {
    PredGradArgs ga;
    memset(&ga, 0, sizeof(ga));
    ga.xs_r = r.xs;
    ga.zpt_r = r.zpt;
    ga.zs_r = r.zs;
    ga.xs_c = c.xs;
    ga.zpt_c = c.zpt;
    ga.zs_c = c.zs;
    ga.alpha = alpha;
    ga.V = V;
    ga.ldv = ldv;
    ga.n_r = r.n;
    ga.n_c = c.n;
    ga.dq = h->dq;
    ga.dqp = h->dqp;
    ga.dz = h->dz;
    ga.n_pass = h->n_pass;
    ga.part_m = part_m;
    ga.part_v = part_v;
    ga.ldp = ldp;
    CK(launch_predict_grad(ga, h->kernel, r.tiles, c.tiles, h->st));
    return GPP_OK;
}

// gpp_predict, gpp_predict_grad (d_mean / d_var) and gpp_acq_argmax (acq): m rows in chunks of mc_alloc rows, of g_step
// rows with the gradient
static int predict_rows(gpp_handle* h, long long m, const Rows& r, double* mean, double* var, AcqSpec* acq,
                        double* d_mean, double* d_var) {
    int rc = check_rows(h, "predict", nullptr, m, r.xq, r.level_idx);
    if (rc != GPP_OK || m <= 0) return rc;
    if (acq && (acq->n_cost <= 0 || !acq->cost || !acq->kind_by_cost || !acq->best_f))
        ARG_FAIL("acq: cost tables missing");
    const bool grad = d_mean || d_var;
    CK(cudaSetDevice(h->device));
    if ((rc = ensure_chunk_buffers(h, m)) != GPP_OK) return rc;
    if (grad && (rc = ensure_grad_buffers(h)) != GPP_OK) return rc;
    if (acq) {
        CK(h->acq_par.reserve(2 * acq->n_cost, h->st));
        CK(h->acq_kind.reserve(acq->n_cost, h->st));
        CK(cudaMemcpyAsync(h->acq_par, acq->cost, sizeof(double) * acq->n_cost, cudaMemcpyDefault, h->st));
        CK(cudaMemcpyAsync(h->acq_par + acq->n_cost, acq->best_f, sizeof(double) * acq->n_cost, cudaMemcpyDefault,
                           h->st));
        CK(cudaMemcpyAsync(h->acq_kind, acq->kind_by_cost, sizeof(int) * acq->n_cost, cudaMemcpyDefault, h->st));
    }
    std::vector<double> hb;
    std::vector<long long> hi;
    const long long step = grad ? h->g_step : h->mc_alloc;
    for (long long base = 0; base < m; base += step) {
        const long long mc = std::min(step, m - base);
        if (h->dq > 0)
            CK(cudaMemcpyAsync(h->c_xq, r.xq + base * h->dq, sizeof(double) * mc * h->dq, cudaMemcpyDefault, h->st));
        if (h->dz > 0) CK(cudaMemcpyAsync(h->c_lvl, r.level_idx + base, sizeof(int) * mc, cudaMemcpyDefault, h->st));
        if (r.noise_idx)
            CK(cudaMemcpyAsync(h->c_noise, r.noise_idx + base, sizeof(int) * mc, cudaMemcpyDefault, h->st));
        if (r.mean_idx) CK(cudaMemcpyAsync(h->c_mean, r.mean_idx + base, sizeof(int) * mc, cudaMemcpyDefault, h->st));
        if (acq && acq->cost_idx)
            CK(cudaMemcpyAsync(h->c_cost, acq->cost_idx + base, sizeof(int) * mc, cudaMemcpyDefault, h->st));
        if ((rc = chunk_front(h, r, base, mc, nullptr, grad ? h->g_U.p : nullptr, acq)) != GPP_OK) return rc;
        const int nblk = (int)((mc + 255) / 256);
        if (grad) {  // V = U L^-1 over the K* chunk, which is not read again, then the gradient partials and their sums
            const Panels rows = chunk_panels(h, mc);
            if ((rc = v_gemm(h, h->g_U, h->c_K, rows.tiles)) != GPP_OK) return rc;
            if ((rc = grad_tiles(h, rows, training_panels(h), h->alpha, h->c_K, h->np, h->g_part_m, h->g_part_v,
                                 step)) != GPP_OK)
                return rc;
            PredGradFinishArgs gf;
            memset(&gf, 0, sizeof(gf));
            gf.part_m = h->g_part_m;
            gf.part_v = h->g_part_v;
            gf.ldp = step;
            gf.rowsq = h->c_rowsq;
            gf.ldr = h->mc_alloc;
            gf.tiles_c = h->T;
            gf.m = (int)mc;
            gf.dq = h->dq;
            gf.w = hyp_w(h);
            gf.sf2 = h->sf2;
            gf.noise_idx = r.noise_idx ? h->c_noise.p : nullptr;
            gf.noise = hyp_noise(h);
            gf.n_noise = h->n_noise;
            gf.include_noise = r.include_noise;
            gf.min_var = r.min_var;
            gf.d_mean = h->g_dmean;
            gf.d_var = h->g_dvar;
            predict_grad_finish_kernel<<<nblk, 256, 0, h->st>>>(gf);
            CK(cudaGetLastError());
            count_launch();
            const size_t gb = sizeof(double) * (size_t)mc * h->dq;
            if (d_mean) CK(cudaMemcpyAsync(d_mean + base * h->dq, h->g_dmean, gb, cudaMemcpyDefault, h->st));
            if (d_var) CK(cudaMemcpyAsync(d_var + base * h->dq, h->g_dvar, gb, cudaMemcpyDefault, h->st));
        }
        if (mean) CK(cudaMemcpyAsync(mean + base, h->c_mu, sizeof(double) * mc, cudaMemcpyDefault, h->st));
        if (var) CK(cudaMemcpyAsync(var + base, h->c_var, sizeof(double) * mc, cudaMemcpyDefault, h->st));
        if (acq) {
            if (acq->scores)
                CK(cudaMemcpyAsync(acq->scores + base, h->c_score, sizeof(double) * mc, cudaMemcpyDefault, h->st));
            hb.resize(nblk);
            hi.resize(nblk);
            CK(cudaMemcpyAsync(hb.data(), h->c_blk_best, sizeof(double) * nblk, cudaMemcpyDeviceToHost, h->st));
            CK(cudaMemcpyAsync(hi.data(), h->c_blk_idx, sizeof(long long) * nblk, cudaMemcpyDeviceToHost, h->st));
        }
        CK(cudaStreamSynchronize(h->st));
        if (acq) {
            for (int b = 0; b < nblk; b++) {
                if (acq->best_index < 0 || hb[b] > acq->best_score ||
                    (hb[b] == acq->best_score && hi[b] < acq->best_index)) {
                    acq->best_score = hb[b];
                    acq->best_index = hi[b];
                }
            }
        }
    }
    return GPP_OK;
}

extern "C" int gpp_predict(gpp_handle* h, int64_t m, const double* xq, const int32_t* level_idx,
                           const int32_t* noise_idx, const int32_t* mean_idx, int include_noise, double min_var,
                           double* mean, double* var) {
    if (!h) ARG_FAIL("gpp_predict: null handle");
    const Rows r = {xq, level_idx, noise_idx, mean_idx, include_noise, min_var};
    return predict_rows(h, m, r, mean, var, nullptr, nullptr, nullptr);
}

extern "C" int gpp_predict_grad(gpp_handle* h, int64_t m, const double* xq, const int32_t* level_idx,
                                const int32_t* noise_idx, const int32_t* mean_idx, int include_noise, double min_var,
                                double* mean, double* var, double* d_mean, double* d_var) {
    if (!h) ARG_FAIL("gpp_predict_grad: null handle");
    // no quantitative input (or no gradient asked for): nothing to differentiate, the gpp_predict sequence
    const bool grad = h->dq > 0 && (d_mean || d_var);
    const Rows r = {xq, level_idx, noise_idx, mean_idx, include_noise, min_var};
    return predict_rows(h, m, r, mean, var, nullptr, grad ? d_mean : nullptr, grad ? d_var : nullptr);
}

extern "C" int gpp_acq_argmax(gpp_handle* h, int64_t m, const double* xq, const int32_t* level_idx,
                              const int32_t* mean_idx, const int32_t* cost_idx, int32_t n_cost, const double* cost,
                              const int32_t* kind_by_cost, const double* best_f, int maximize, double si,
                              double y_min, double y_std, double min_var, double* scores, double* best_score,
                              int64_t* best_index) {
    if (!h) ARG_FAIL("gpp_acq_argmax: null handle");
    AcqSpec a;
    a.cost_idx = cost_idx;
    a.n_cost = n_cost;
    a.cost = cost;
    a.kind_by_cost = kind_by_cost;
    a.best_f = best_f;
    a.maximize = maximize;
    a.si = si;
    a.y_min = y_min;
    a.y_std = y_std;
    a.scores = scores;
    // the reference's candidate-table branch predicts with include_noise=False (BO_GP_plus.py:185-186)
    const Rows r = {xq, level_idx, nullptr, mean_idx, 0, min_var};
    int rc = predict_rows(h, m, r, nullptr, nullptr, &a, nullptr, nullptr);
    if (rc != GPP_OK) return rc;
    if (best_score) *best_score = a.best_score;
    if (best_index) *best_index = a.best_index;
    return GPP_OK;
}

// Loads m points into the set s: their inputs and panels once (ld mp = m padded to 128), then the prediction chunk loop
// on the set's panels with U = K* L^-T of every row stored in s.U (rows >= m come out zero).  Mean and variance of row
// i go to mean[i] / var[i] when given, the rows' noise groups to noise_out when the variance includes noise.
static int load_point_set(gpp_handle* h, PointSet& s, long long m, const Rows& r, int* noise_out, double* mean,
                          double* var) {
    const long long mp = round128(m);
    CK(s.xq.reserve(mp * std::max(h->dq, 1), h->st));
    CK(s.xs.reserve(mp * h->dqp, h->st));
    CK(s.nrm.reserve(mp, h->st));
    CK(s.zpt.reserve(mp * ZP * h->n_pass, h->st));
    CK(s.U.reserve(mp * h->np, h->st));
    CK(s.lvl.reserve(mp, h->st));
    s.mp = mp;
    if (h->dq > 0) CK(cudaMemcpyAsync(s.xq, r.xq, sizeof(double) * m * h->dq, cudaMemcpyDefault, h->st));
    if (h->dz > 0) CK(cudaMemcpyAsync(s.lvl, r.level_idx, sizeof(int) * m, cudaMemcpyDefault, h->st));
    if (noise_out && r.include_noise && r.noise_idx)
        CK(cudaMemcpyAsync(noise_out, r.noise_idx, sizeof(int) * m, cudaMemcpyDefault, h->st));
    int rc = prep_panels(h, s.xq, h->dz > 0 ? s.lvl.p : nullptr, m, mp, s.xs, nullptr, s.nrm, s.zpt);
    if (rc != GPP_OK) return rc;
    for (long long base = 0; base < m; base += h->mc_alloc) {
        const long long mc = std::min(h->mc_alloc, m - base);
        if (r.noise_idx)
            CK(cudaMemcpyAsync(h->c_noise, r.noise_idx + base, sizeof(int) * mc, cudaMemcpyDefault, h->st));
        if (r.mean_idx) CK(cudaMemcpyAsync(h->c_mean, r.mean_idx + base, sizeof(int) * mc, cudaMemcpyDefault, h->st));
        const Panels rows = {s.xs + base * h->dqp, s.nrm + base, s.zpt + base * ZP, mp * ZP, (int)mc,
                             (int)(round128(mc) / CT)};
        if ((rc = chunk_front(h, r, base, mc, &rows, s.U + base * h->np, nullptr)) != GPP_OK) return rc;
        if (mean) CK(cudaMemcpyAsync(mean + base, h->c_mu, sizeof(double) * mc, cudaMemcpyDefault, h->st));
        if (var) CK(cudaMemcpyAsync(var + base, h->c_var, sizeof(double) * mc, cudaMemcpyDefault, h->st));
        CK(cudaStreamSynchronize(h->st));
    }
    // Columns n .. Np of U are K* L^-T against the identity padding of K_y, i.e. zero in exact arithmetic; clear them
    // so that products over whole 128-blocks of U never depend on how L^-1's padding was produced.
    if (h->np > h->n)
        CK(cudaMemset2DAsync(s.U + h->n, sizeof(double) * h->np, 0, sizeof(double) * (h->np - h->n), (size_t)mp, h->st));
    return GPP_OK;
}

// ---------------------------------------------------------------------------------------------
// Joint posterior over m candidates: Sigma* = K** - K* K_y^-1 K*^T = K** - U U^T with U = K* L^-T, and draws
// mu + E L*^T with L* L*^T = Sigma* + jitter I.  Stages (all on h->st, none of them touches A, M, S, alpha or the
// captured graphs):
//   J1  the joint set (load_point_set; mean bitwise gpp_predict's)
//   J2  K** on the lower tiles (+ noise, + jitter), then Sigma* -= U U^T over K range [0, T)  (one DMMA SYRK)
//   J3  potrf_blocked(Sigma*) in DMMA arithmetic whatever the handle's FP64 mode, psd_safe_cholesky ladder
//   J4  per chunk of base samples: Y = mu + E L*^T  (one triangular DMMA GEMM)

// joint-only buffers for mp rows.  The draw chunk (up to 2 x 1 GiB) is released when the joint set is about to grow,
// so that it is not held while the larger set is allocated; the next gpp_sample_posterior allocates it again.
static int ensure_joint_buffers(gpp_handle* h, long long mp) {
    if (mp > (long long)h->jset.nrm.cap) {  // (nrm holds one double per row of the set)
        CK(cudaStreamSynchronize(h->st));
        h->j_E.release();
        h->j_Y.release();
    }
    CK(h->j_S.reserve(mp * mp, h->st));
    CK(h->j_Minv.reserve(mp * mp, h->st));
    CK(h->j_diag.reserve(mp, h->st));
    CK(h->j_mu.reserve(mp, h->st, true));
    CK(h->j_logdet.reserve(mp / 128, h->st));
    CK(h->j_noise.reserve(mp, h->st));
    CK(h->j_info.reserve(1, h->st));
    return GPP_OK;
}

static const char* joint_count_err(long long m) {
    return (m < 0 || m > GPP_MAX_JOINT) ? "m must be in [0, GPP_MAX_JOINT]" : nullptr;
}

// J1: the joint set, the predictive mean into j_mu
static int joint_stage_u(gpp_handle* h, long long m, const Rows& r) {
    CK(cudaSetDevice(h->device));
    int rc = ensure_chunk_buffers(h, m);  // before the joint buffers: a handle holding them has mc_alloc > 0
    if (rc != GPP_OK || (rc = ensure_joint_buffers(h, round128(m))) != GPP_OK) return rc;
    return load_point_set(h, h->jset, m, r, h->j_noise, h->j_mu, nullptr);
}

// J2: Sigma* (lower tiles) = K** + diag(noise + jitter) - U U^T into j_S
static int joint_stage_sigma(gpp_handle* h, long long m, const int32_t* noise_idx, int include_noise, double jitter) {
    const long long mp = round128(m);
    const int mt = (int)(mp / 128);
    joint_diag_kernel<<<(int)((mp + 255) / 256), 256, 0, h->st>>>(noise_idx ? h->j_noise.p : nullptr, hyp_noise(h),
                                                                 h->n_noise, include_noise, jitter, (int)m, (int)mp,
                                                                 h->j_diag);
    CK(cudaGetLastError());
    count_launch();
    CovArgs ca;
    memset(&ca, 0, sizeof(ca));
    ca.out = h->j_S;
    ca.ld = mp;
    ca.tri = 1;
    ca.same = 1;
    ca.pad_identity = 1;
    ca.diag_add = h->j_diag;
    const Panels set = {h->jset.xs, h->jset.nrm, h->jset.zpt, mp * ZP, (int)m, mt};
    int rc = launch_cov_passes(h, ca, set, set);
    if (rc != GPP_OK) return rc;
    GemmOp op = gemm_default();  // Sigma* -= U U^T on the lower tiles (the trailing_update op shape)
    op.A = h->jset.U;
    op.lda = (int)h->np;
    op.B = h->jset.U;
    op.ldb = (int)h->np;
    op.C = h->j_S;
    op.ldc = (int)mp;
    op.map = MAP_TRI;
    op.tiles_m = op.tiles_m_last = mt;
    op.tiles_n = mt;
    op.klo_c = 0;
    op.khi_c = h->T;
    op.alpha = -1.0;
    op.beta = 1.0;
    CK(launch_gemm(op, true, true, 1, h->st));
    return GPP_OK;
}

extern "C" int gpp_predict_joint(gpp_handle* h, int64_t m, const double* xq, const int32_t* level_idx,
                                 const int32_t* noise_idx, const int32_t* mean_idx, int include_noise, double* mean,
                                 double* cov) {
    int rc = check_rows(h, "gpp_predict_joint", joint_count_err(m), m, xq, level_idx);
    if (rc != GPP_OK || m == 0) return rc;
    const Rows r = {xq, level_idx, noise_idx, mean_idx, include_noise, 0.0};
    if ((rc = joint_stage_u(h, m, r)) != GPP_OK) return rc;
    if ((rc = joint_stage_sigma(h, m, noise_idx, include_noise, 0.0)) != GPP_OK) return rc;
    const long long mp = round128(m);
    const int nb = (int)(mp / 32);
    mirror_lower_kernel<<<dim3(nb, nb), dim3(32, 8), 0, h->st>>>(h->j_S, mp);
    CK(cudaGetLastError());
    count_launch();
    if (mean) CK(cudaMemcpyAsync(mean, h->j_mu, sizeof(double) * m, cudaMemcpyDefault, h->st));
    if (cov)
        CK(cudaMemcpy2DAsync(cov, sizeof(double) * m, h->j_S, sizeof(double) * mp, sizeof(double) * m, (size_t)m,
                             cudaMemcpyDefault, h->st));
    CK(cudaStreamSynchronize(h->st));
    return GPP_OK;
}

extern "C" int gpp_sample_posterior(gpp_handle* h, int64_t m, const double* xq, const int32_t* level_idx,
                                    const int32_t* noise_idx, const int32_t* mean_idx, int include_noise,
                                    int64_t n_samples, const double* base_samples, double* samples, double* jitter) {
    int rc = check_rows(h, "gpp_sample_posterior", joint_count_err(m), m, xq, level_idx);
    if (rc != GPP_OK) return rc;
    if (n_samples < 0) ARG_FAIL("gpp_sample_posterior: n_samples must be >= 0");
    if (m > 0 && n_samples > 0 && (!base_samples || !samples)) ARG_FAIL("gpp_sample_posterior: samples missing");
    if (m == 0) {
        if (jitter) *jitter = 0.0;
        return GPP_OK;
    }
    const Rows r = {xq, level_idx, noise_idx, mean_idx, include_noise, 0.0};
    if ((rc = joint_stage_u(h, m, r)) != GPP_OK) return rc;
    const long long mp = round128(m);
    const int mt = (int)(mp / 128);
    // The leaf writes only the lower 32 x 32 sub-blocks of each diagonal block of L*^-1, and the TRSM reads the whole
    // block, so the [mp x mp] matrix potrf_blocked addresses must start at zero.  A previous call with a larger mp
    // left inverse entries there at another leading dimension: clear it on every call.
    CK(cudaMemsetAsync(h->j_Minv, 0, sizeof(double) * mp * mp, h->st));
    int a = 0;
    for (;; a++) {
        if (a == 4) {
            g_err = "gpp_sample_posterior: the joint posterior covariance is not positive definite after adding "
                    "jitter up to 1e-6";
            return GPP_ERR_NOT_PD;
        }
        if ((rc = joint_stage_sigma(h, m, noise_idx, include_noise, kJitter[a])) != GPP_OK) return rc;
        CK(cudaMemsetAsync(h->j_info, 0, sizeof(int), h->st));
        CK(potrf_blocked(h->j_S, h->j_Minv, (int)mp, mt, h->j_logdet, h->j_info, h->st));
        int info = 0;
        CK(cudaMemcpyAsync(&info, h->j_info, sizeof(int), cudaMemcpyDeviceToHost, h->st));
        CK(cudaStreamSynchronize(h->st));
        if (info & 2) {
            g_err = "gpp_sample_posterior: NaN encountered while factorising the joint posterior covariance";
            return GPP_ERR_NAN;
        }
        if (info == 0) break;
    }
    if (jitter) *jitter = kJitter[a];
    zero_diag_upper_kernel<<<mt, 256, 0, h->st>>>(h->j_S, mp);
    CK(cudaGetLastError());
    count_launch();
    if (n_samples == 0) {
        CK(cudaStreamSynchronize(h->st));
        return GPP_OK;
    }
    long long cap = ((1LL << 27) / mp) / 128 * 128;
    if (cap < 128) cap = 128;
    const long long sc = std::min(round128(n_samples), cap);
    // base samples and draws of one chunk, sc x mp doubles each
    CK(h->j_E.reserve(sc * mp, h->st, true));
    CK(h->j_Y.reserve(sc * mp, h->st));
    for (long long s0 = 0; s0 < n_samples; s0 += sc) {
        const long long rows = std::min(sc, n_samples - s0);
        const long long rp = round128(rows);
        CK(cudaMemcpy2DAsync(h->j_E, sizeof(double) * mp, base_samples + s0 * m, sizeof(double) * m,
                             sizeof(double) * m, (size_t)rows, cudaMemcpyDefault, h->st));
        if (mp > m)  // padding columns of E meet only zeros of L*, but must not be stale non-finite values
            CK(cudaMemset2DAsync(h->j_E + m, sizeof(double) * mp, 0, sizeof(double) * (mp - m), (size_t)rp, h->st));
        const long long total = rp * mp;
        fill_rows_kernel<<<(int)std::min<long long>((total + 255) / 256, 4096), 256, 0, h->st>>>(h->j_Y, h->j_mu, mp,
                                                                                                total);
        CK(cudaGetLastError());
        count_launch();
        GemmOp op = gemm_default();  // Y += E L*^T: B(tj, kb) = L*[tj, kb], kb in [0, tj]
        op.A = h->j_E;
        op.lda = (int)mp;
        op.B = h->j_S;
        op.ldb = (int)mp;
        op.C = h->j_Y;
        op.ldc = (int)mp;
        op.tiles_m = op.tiles_m_last = (int)(rp / 128);
        op.tiles_n = mt;
        op.klo_c = 0;
        op.khi_sel = KSEL_TJ;
        op.khi_c = 1;
        op.beta = 1.0;
        CK(launch_gemm(op, true, true, 1, h->st));
        CK(cudaMemcpy2DAsync(samples + s0 * m, sizeof(double) * m, h->j_Y, sizeof(double) * mp, sizeof(double) * m,
                             (size_t)rows, cudaMemcpyDefault, h->st));
    }
    CK(cudaStreamSynchronize(h->st));
    return GPP_OK;
}

// ---------------------------------------------------------------------------------------------
// Joint posteriors of b independent t-batches of q candidates (qbatch.cuh): chunks of whole t-batches through the
// chunk front with U stored, then only the q x q diagonal blocks.  Every 128-row tile of the chunk buffers holds
// qpt = 128 / q whole t-batches followed by padding rows, so chunks (multiples of 128 rows) hold whole t-batches.
struct QBatchSpec {
    long long b;
    int q, qpt;
};

static QBatchSpec qbatch_spec(long long b, int q) { return {b, q, CT / q}; }

static long long qbatch_rows(const QBatchSpec& s) { return (s.b + s.qpt - 1) / s.qpt * CT; }

static const char* qbatch_count_err(long long b, int q) {
    if (q < 1 || q > GPP_MAX_QBATCH) return "q must be in [1, GPP_MAX_QBATCH]";
    return b < 0 ? "b must be >= 0" : nullptr;
}

// one chunk of a t-batch call: rows [base, base + mc), tiles of 128 rows, t-batches [bt0, bt0 + nb)
struct QChunk {
    long long base, mc, mcp, bt0, nb;
    int tiles;
};

static QChunk qbatch_chunk(const QBatchSpec& s, long long base, long long step) {
    QChunk c;
    c.base = base;
    c.mc = std::min(step, qbatch_rows(s) - base);
    c.mcp = round128(c.mc);
    c.tiles = (int)(c.mcp / CT);
    c.bt0 = base / CT * s.qpt;
    c.nb = std::min(s.b, c.bt0 + (long long)c.tiles * s.qpt) - c.bt0;
    return c;
}

// rows of nbat t-batches, from t-batch bt0 of a compact [b*q rows] array, to (into_tiles) or from their tile slots in
// a chunk buffer: one pitched copy for the full tiles, one plain copy for the last, partly filled one
static cudaError_t qb_copy_rows(const QBatchSpec& s, void* dst, const void* src, size_t row_bytes, long long bt0,
                                long long nbat, bool into_tiles, cudaStream_t st) {
    if (row_bytes == 0 || nbat <= 0) return cudaSuccess;
    const size_t run = (size_t)s.qpt * s.q * row_bytes, tile = (size_t)CT * row_bytes;
    const size_t off = (size_t)bt0 * s.q * row_bytes;
    char* d = (char*)dst + (into_tiles ? 0 : off);
    const char* src_c = (const char*)src + (into_tiles ? off : 0);
    const size_t dp = into_tiles ? tile : run, sp = into_tiles ? run : tile;
    const long long full = nbat / s.qpt, rest = nbat % s.qpt;
    if (full > 0) {
        cudaError_t e = cudaMemcpy2DAsync(d, dp, src_c, sp, run, (size_t)full, cudaMemcpyDefault, st);
        if (e != cudaSuccess) return e;
    }
    if (rest > 0)
        return cudaMemcpyAsync(d + full * dp, src_c + full * sp, (size_t)rest * s.q * row_bytes, cudaMemcpyDefault,
                               st);
    return cudaSuccess;
}

// chunk, gradient and q x q block buffers of a t-batch call.  q_buf is sized at g_step * q: when g_step has grown since
// its allocation (q_gm, sized at g_step, shows it) it is allocated afresh rather than kept at an older chunk's size.
static int qbatch_setup(gpp_handle* h, const QBatchSpec& s) {
    CK(cudaSetDevice(h->device));
    int rc = ensure_chunk_buffers(h, qbatch_rows(s));
    if (rc != GPP_OK || (rc = ensure_grad_buffers(h)) != GPP_OK) return rc;
    if (h->q_gm.cap < (size_t)h->g_step) h->q_buf.release();
    CK(h->q_buf.reserve(h->g_step * s.q, h->st));
    CK(h->q_gm.reserve(h->g_step, h->st));
    return GPP_OK;
}

// the rows of the chunk's t-batches into their tile slots (padding rows are zero points of level, group and mean 0),
// then the chunk front with U stored in g_U
static int qbatch_front(gpp_handle* h, const QBatchSpec& s, const Rows& r, const QChunk& c) {
    CK(cudaMemsetAsync(h->c_xq, 0, sizeof(double) * c.mcp * h->dq, h->st));
    CK(cudaMemsetAsync(h->c_lvl, 0, sizeof(int) * c.mcp, h->st));
    CK(cudaMemsetAsync(h->c_noise, 0, sizeof(int) * c.mcp, h->st));
    CK(cudaMemsetAsync(h->c_mean, 0, sizeof(int) * c.mcp, h->st));
    CK(qb_copy_rows(s, h->c_xq, r.xq, sizeof(double) * h->dq, c.bt0, c.nb, true, h->st));
    if (h->dz > 0) CK(qb_copy_rows(s, h->c_lvl, r.level_idx, sizeof(int), c.bt0, c.nb, true, h->st));
    if (r.noise_idx) CK(qb_copy_rows(s, h->c_noise, r.noise_idx, sizeof(int), c.bt0, c.nb, true, h->st));
    if (r.mean_idx) CK(qb_copy_rows(s, h->c_mean, r.mean_idx, sizeof(int), c.bt0, c.nb, true, h->st));
    return chunk_front(h, r, c.base, c.mc, nullptr, h->g_U, nullptr);
}

// Sigma_t = K**_t - U_t U_t^T of the chunk's t-batches into q_buf
static int qbatch_sigma(gpp_handle* h, const QBatchSpec& s, const Rows& r, const QChunk& c) {
    QSyrkArgs sa;
    memset(&sa, 0, sizeof(sa));
    sa.U = h->g_U;
    sa.ldu = h->np;
    sa.kcols = (int)h->n;
    sa.rowsq = h->c_rowsq;
    sa.ldr = h->mc_alloc;
    sa.tiles_c = h->T;
    sa.xs = h->c_xs;
    sa.zpt = h->c_zpt;
    sa.zs = c.mcp * ZP;
    sa.dq = h->dq;
    sa.dqp = h->dqp;
    sa.dz = h->dz;
    sa.n_pass = h->n_pass;
    sa.sf2 = h->sf2;
    sa.noise_idx = r.noise_idx ? h->c_noise.p : nullptr;
    sa.noise = hyp_noise(h);
    sa.n_noise = h->n_noise;
    sa.include_noise = r.include_noise;
    sa.q = s.q;
    sa.qpt = s.qpt;
    sa.nb = c.nb;
    sa.cov = h->q_buf;
    CK(launch_qbatch_syrk(sa, h->kernel, c.tiles, h->st));
    return GPP_OK;
}

// Backward, first step after V = U L^-1 (in c_K): W = blockdiag(G + G^T) V into g_U (U is not read again), G_t in q_buf
static int qbatch_w(gpp_handle* h, const QBatchSpec& s, const QChunk& c) {
    QWArgs wa;
    wa.V = h->c_K;
    wa.ldv = h->np;
    wa.G = h->q_buf;
    wa.q = s.q;
    wa.qpt = s.qpt;
    wa.nb = c.nb;
    wa.W = h->g_U;
    wa.ldw = h->np;
    qbatch_w_kernel<<<dim3((unsigned)(h->np / QB_KC), (unsigned)c.tiles), QB_THREADS, 0, h->st>>>(wa);
    CK(cudaGetLastError());
    count_launch();
    return GPP_OK;
}

// Backward, last step: the in-batch K**_t term, then d_xq of the chunk's rows from the gradient partials over tiles_c
// column tiles (tile layout in g_dvar), gathered to the caller's rows; g_mean: the upstream mean gradient in the tile
// layout, or NULL
static int qbatch_grad_finish(gpp_handle* h, const QBatchSpec& s, const QChunk& c, const double* part_m,
                              const double* part_v, long long ldp, int tiles_c, const double* g_mean, double* d_xq) {
    QInArgs ia;
    ia.xs = h->c_xs;
    ia.zpt = h->c_zpt;
    ia.zs = c.mcp * ZP;
    ia.dq = h->dq;
    ia.dqp = h->dqp;
    ia.dz = h->dz;
    ia.n_pass = h->n_pass;
    ia.G = h->q_buf;
    ia.q = s.q;
    ia.qpt = s.qpt;
    ia.nb = c.nb;
    ia.rows = (int)c.mcp;
    ia.part_k = h->g_dmean;
    CK(launch_qbatch_inbatch_grad(ia, h->kernel, h->st));
    QFinishArgs qf;
    qf.part_m = part_m;
    qf.part_v = part_v;
    qf.ldp = ldp;
    qf.tiles_c = tiles_c;
    qf.part_k = h->g_dmean;
    qf.g_mean = g_mean;
    qf.m = (int)c.mcp;
    qf.dq = h->dq;
    qf.w = hyp_w(h);
    qf.sf2 = h->sf2;
    qf.d_x = h->g_dvar;
    qbatch_grad_finish_kernel<<<(int)((c.mcp + 255) / 256), 256, 0, h->st>>>(qf);
    CK(cudaGetLastError());
    count_launch();
    CK(qb_copy_rows(s, d_xq, h->g_dvar, sizeof(double) * h->dq, c.bt0, c.nb, false, h->st));
    return GPP_OK;
}

// the status word of a gpp_acq_qbatch / gpp_nipv_qbatch / gpp_kg_qbatch / gpp_gibbon_qbatch chunk, once the chunk has
// finished
static int qbatch_status(gpp_handle* h, const char* name, const char* nan_msg) {
    int info = 0;
    CK(cudaMemcpyAsync(&info, h->a_info, sizeof(int), cudaMemcpyDeviceToHost, h->st));
    CK(cudaStreamSynchronize(h->st));
    if (info & 2) {
        g_err = nan_msg;
        return GPP_ERR_NAN;
    }
    if (info & 1) {
        g_err = std::string(name) +
                ": a t-batch posterior covariance is not positive definite after adding jitter up to 1e-6";
        return GPP_ERR_NOT_PD;
    }
    return GPP_OK;
}

// values, jitters and the status word of gpp_acq_qbatch / gpp_nipv_qbatch / gpp_kg_qbatch / gpp_gibbon_qbatch (a chunk
// holds at most g_step t-batches), and the base samples (max values) of the call (e_elems doubles)
static int ensure_acq_buffers(gpp_handle* h, long long e_elems) {
    CK(h->a_info.reserve(1, h->st));
    CK(h->a_E.reserve(e_elems, h->st));
    CK(h->a_val.reserve(h->g_step, h->st));
    CK(h->a_jit.reserve(h->g_step, h->st));
    return GPP_OK;
}

extern "C" int gpp_posterior_qbatch(gpp_handle* h, int64_t b, int32_t q, const double* xq, const int32_t* level_idx,
                                    const int32_t* noise_idx, const int32_t* mean_idx, int include_noise,
                                    double* mean, double* cov) {
    int rc = check_rows(h, "gpp_posterior_qbatch", qbatch_count_err(b, q), b, xq, level_idx);
    if (rc != GPP_OK || b == 0) return rc;
    const QBatchSpec s = qbatch_spec(b, q);
    const Rows r = {xq, level_idx, noise_idx, mean_idx, include_noise, 0.0};
    if ((rc = qbatch_setup(h, s)) != GPP_OK) return rc;
    for (long long base = 0; base < qbatch_rows(s); base += h->g_step) {
        const QChunk c = qbatch_chunk(s, base, h->g_step);
        if ((rc = qbatch_front(h, s, r, c)) != GPP_OK) return rc;
        if (cov) {
            if ((rc = qbatch_sigma(h, s, r, c)) != GPP_OK) return rc;
            const size_t qq = (size_t)q * q;
            CK(cudaMemcpyAsync(cov + c.bt0 * qq, h->q_buf, sizeof(double) * c.nb * qq, cudaMemcpyDefault, h->st));
        }
        if (mean) CK(qb_copy_rows(s, mean, h->c_mu, sizeof(double), c.bt0, c.nb, false, h->st));
        CK(cudaStreamSynchronize(h->st));
    }
    return GPP_OK;
}

extern "C" int gpp_posterior_qbatch_grad(gpp_handle* h, int64_t b, int32_t q, const double* xq,
                                         const int32_t* level_idx, const int32_t* noise_idx, const int32_t* mean_idx,
                                         int include_noise, const double* g_mean, const double* g_cov, double* d_xq) {
    int rc = check_rows(h, "gpp_posterior_qbatch_grad", qbatch_count_err(b, q), b, xq, level_idx);
    if (rc != GPP_OK) return rc;
    if (b > 0 && h->dq > 0 && !d_xq) ARG_FAIL("gpp_posterior_qbatch_grad: d_xq missing");
    if (b == 0 || h->dq == 0) return GPP_OK;  // no quantitative input: d_xq is empty
    const QBatchSpec s = qbatch_spec(b, q);
    const Rows r = {xq, level_idx, noise_idx, mean_idx, include_noise, 0.0};
    if ((rc = qbatch_setup(h, s)) != GPP_OK) return rc;
    const long long step = h->g_step;
    for (long long base = 0; base < qbatch_rows(s); base += step) {
        const QChunk c = qbatch_chunk(s, base, step);
        if ((rc = qbatch_front(h, s, r, c)) != GPP_OK) return rc;
        if ((rc = v_gemm(h, h->g_U, h->c_K, c.tiles)) != GPP_OK) return rc;
        const size_t qq = (size_t)q * q;
        if (g_cov)
            CK(cudaMemcpyAsync(h->q_buf, g_cov + c.bt0 * qq, sizeof(double) * c.nb * qq, cudaMemcpyDefault, h->st));
        else
            CK(cudaMemsetAsync(h->q_buf, 0, sizeof(double) * c.nb * qq, h->st));
        if (g_mean) {
            CK(cudaMemsetAsync(h->q_gm, 0, sizeof(double) * c.mcp, h->st));
            CK(qb_copy_rows(s, h->q_gm, g_mean, sizeof(double), c.bt0, c.nb, true, h->st));
        }
        if ((rc = qbatch_w(h, s, c)) != GPP_OK) return rc;
        if ((rc = grad_tiles(h, chunk_panels(h, c.mc), training_panels(h), h->alpha, h->g_U, h->np, h->g_part_m,
                             h->g_part_v, step)) != GPP_OK)
            return rc;
        if ((rc = qbatch_grad_finish(h, s, c, h->g_part_m, h->g_part_v, step, h->T, g_mean ? h->q_gm.p : nullptr,
                                     d_xq)) != GPP_OK)
            return rc;
        CK(cudaStreamSynchronize(h->st));
    }
    return GPP_OK;
}

// ---------------------------------------------------------------------------------------------
// Monte-Carlo batch acquisition (qacq.cuh): the gpp_posterior_qbatch chunks, then per t-batch the factor, the samples
// and the utility in one CTA; with d_xq, the utility's adjoint (G_t, mu_bar) feeds the q-batch backward in the same
// chunk, so no block leaves the device.

// the utility, its parameters in scaled units and the per-t-batch outputs
struct QAcqSpec {
    int kind, n_base, maximize;
    double best_f, cbeta;
    long long S;
    const double* E;  // [S*q] caller's base samples
    double* values;   // [b]
    double* jitter;   // [b] or NULL
};

// values and jitters of the chunk's t-batches from Sigma_t in q_buf; with the gradient, G_t over Sigma_t in q_buf and
// mu_bar into q_gm
static int qbatch_mc(gpp_handle* h, const QBatchSpec& s, const QAcqSpec& a, const QChunk& c, bool grad) {
    if (grad) CK(cudaMemsetAsync(h->q_gm, 0, sizeof(double) * c.mcp, h->st));
    QAcqArgs aa;
    memset(&aa, 0, sizeof(aa));
    aa.blk = h->q_buf;
    aa.mu = h->c_mu;
    aa.gm = h->q_gm;
    aa.E = h->a_E;
    aa.S = a.S;
    aa.q = s.q;
    aa.qpt = s.qpt;
    aa.n_base = a.n_base;
    aa.nb = c.nb;
    aa.sgn = a.maximize ? 1.0 : -1.0;
    aa.best_f = a.best_f;
    aa.cbeta = a.cbeta;
    aa.grad = grad ? 1 : 0;
    aa.value = h->a_val;
    aa.jitter = h->a_jit;
    aa.info = h->a_info;
    CK(launch_qacq(aa, a.kind, h->st));
    CK(cudaMemcpyAsync(a.values + c.bt0, h->a_val, sizeof(double) * c.nb, cudaMemcpyDefault, h->st));
    if (a.jitter) CK(cudaMemcpyAsync(a.jitter + c.bt0, h->a_jit, sizeof(double) * c.nb, cudaMemcpyDefault, h->st));
    return GPP_OK;
}

extern "C" int gpp_acq_qbatch(gpp_handle* h, int64_t b, int32_t q_tot, const double* xq, const int32_t* level_idx,
                              const int32_t* noise_idx, const int32_t* mean_idx, int include_noise, int kind,
                              int32_t n_baseline, double best_f, double beta, int maximize, int64_t n_samples,
                              const double* base_samples, double* values, double* d_xq, double* jitter) {
    int rc = check_rows(h, "gpp_acq_qbatch", qbatch_count_err(b, q_tot), b, xq, level_idx);
    if (rc != GPP_OK) return rc;
    if (kind != GPP_QACQ_EI && kind != GPP_QACQ_NEI && kind != GPP_QACQ_UCB) ARG_FAIL("gpp_acq_qbatch: unknown kind");
    if (kind == GPP_QACQ_NEI ? (n_baseline < 1 || n_baseline >= q_tot) : n_baseline != 0)
        ARG_FAIL("gpp_acq_qbatch: n_baseline must be in [1, q_tot) for GPP_QACQ_NEI and 0 otherwise");
    if (n_samples < 1 || n_samples > GPP_MAX_MC_SAMPLES)
        ARG_FAIL("gpp_acq_qbatch: n_samples must be in [1, GPP_MAX_MC_SAMPLES]");
    if (!base_samples || !values) ARG_FAIL("gpp_acq_qbatch: base_samples / values missing");
    if (kind == GPP_QACQ_UCB && !(beta >= 0.0 && beta < INFINITY))
        ARG_FAIL("gpp_acq_qbatch: beta must be finite and >= 0");
    if (b == 0) return GPP_OK;
    QAcqSpec a;
    memset(&a, 0, sizeof(a));
    a.kind = kind;
    a.n_base = kind == GPP_QACQ_NEI ? n_baseline : 0;
    a.maximize = maximize;
    a.best_f = best_f;
    a.cbeta = sqrt(beta * M_PI / 2.0);
    a.S = n_samples;
    a.E = base_samples;
    a.values = values;
    a.jitter = jitter;
    const QBatchSpec s = qbatch_spec(b, q_tot);
    const Rows r = {xq, level_idx, noise_idx, mean_idx, include_noise, 0.0};
    const bool grad = d_xq && h->dq > 0;
    if ((rc = qbatch_setup(h, s)) != GPP_OK || (rc = ensure_acq_buffers(h, a.S * s.q)) != GPP_OK) return rc;
    CK(cudaMemcpyAsync(h->a_E, a.E, sizeof(double) * a.S * s.q, cudaMemcpyDefault, h->st));
    CK(cudaMemsetAsync(h->a_info, 0, sizeof(int), h->st));
    const long long step = h->g_step;
    for (long long base = 0; base < qbatch_rows(s); base += step) {
        const QChunk c = qbatch_chunk(s, base, step);
        if ((rc = qbatch_front(h, s, r, c)) != GPP_OK || (rc = qbatch_sigma(h, s, r, c)) != GPP_OK ||
            (rc = qbatch_mc(h, s, a, c, grad)) != GPP_OK)
            return rc;
        if (grad) {  // G_t is in q_buf and mu_bar in q_gm already
            if ((rc = v_gemm(h, h->g_U, h->c_K, c.tiles)) != GPP_OK || (rc = qbatch_w(h, s, c)) != GPP_OK) return rc;
            if ((rc = grad_tiles(h, chunk_panels(h, c.mc), training_panels(h), h->alpha, h->g_U, h->np, h->g_part_m,
                                 h->g_part_v, step)) != GPP_OK)
                return rc;
            if ((rc = qbatch_grad_finish(h, s, c, h->g_part_m, h->g_part_v, step, h->T, h->q_gm, d_xq)) != GPP_OK)
                return rc;
        }
        if ((rc = qbatch_status(h, "gpp_acq_qbatch", "gpp_acq_qbatch: NaN in a t-batch posterior or its samples")) !=
            GPP_OK)
            return rc;
    }
    return GPP_OK;
}

// ---------------------------------------------------------------------------------------------
// Batch integrated posterior variance (nipv.cuh): gpp_ipv_points keeps the integration set's panels, U_I and V_I on the
// handle for the current factor; gpp_nipv_qbatch runs the gpp_posterior_qbatch chunks with the candidates' noise,
// forms C^T against the set, and feeds the closed form's adjoint to the q-batch backward in the same chunk.
static bool ipv_valid(const gpp_handle* h) { return h->factorized && h->i_m > 0 && h->i_gen == h->fgen; }

// rows of one gpp_nipv_qbatch chunk: the C^T buffer [rows x mp of the set] holds at most 2^27 doubles (1 GiB)
static long long nipv_step(const gpp_handle* h) {
    return std::min(h->g_step, std::max(128LL, ((1LL << 27) / h->iset.mp) / 128 * 128));
}

static Panels ipv_panels(const gpp_handle* h) {
    return {h->iset.xs, h->iset.nrm, h->iset.zpt, h->iset.mp * ZP, (int)h->i_m, (int)(h->iset.mp / CT)};
}

extern "C" int gpp_ipv_points(gpp_handle* h, int64_t m, const double* xq, const int32_t* level_idx) {
    int rc = check_rows(h, "gpp_ipv_points", (m < 1 || m > GPP_MAX_IPV_POINTS) ? "m must be in [1, GPP_MAX_IPV_POINTS]"
                                                                               : nullptr,
                        m, xq, level_idx);
    if (rc != GPP_OK) return rc;
    CK(cudaSetDevice(h->device));
    h->i_m = 0;  // no valid set until this call has finished
    const long long mp = round128(m);
    if ((rc = ensure_chunk_buffers(h, m)) != GPP_OK) return rc;
    CK(h->i_V.reserve(mp * h->np, h->st));
    CK(h->i_zero.reserve(mp, h->st, true));
    // U_I through the prediction chunk loop; v_m = sf2 - |U_m|^2 unclamped and without noise
    std::vector<double> v((size_t)m);
    const Rows r = {xq, level_idx, nullptr, nullptr, 0, -INFINITY};
    if ((rc = load_point_set(h, h->iset, m, r, nullptr, nullptr, v.data())) != GPP_OK) return rc;
    if ((rc = v_gemm(h, h->iset.U, h->i_V, (int)(mp / CT))) != GPP_OK) return rc;  // V_I = U_I L^-1 = K_I K_y^-1
    CK(cudaStreamSynchronize(h->st));
    double sum = 0.0;
    for (long long i = 0; i < m; i++) sum += v[(size_t)i];
    if (std::isnan(sum)) {
        g_err = "gpp_ipv_points: NaN in the latent variance at the integration points";
        return GPP_ERR_NAN;
    }
    h->i_vbar = sum / (double)m;
    h->i_m = m;
    h->i_gen = h->fgen;
    return GPP_OK;
}

// C^T = K(X_chunk, X_I) - U_chunk U_I^T into n_C, then per t-batch G_t = C_t^T C_t, A_t's factor and the value (A_bar_t
// over A_t in q_buf and -A_t^-1 / M in n_Ai with the gradient)
static int nipv_forward(gpp_handle* h, const QBatchSpec& s, const QChunk& c, double* values, double* jitter,
                        bool grad) {
    const Panels iset = ipv_panels(h);
    CovArgs cc;
    memset(&cc, 0, sizeof(cc));
    cc.out = h->n_C;
    cc.ld = h->iset.mp;
    int rc = launch_cov_passes(h, cc, chunk_panels(h, c.mc), iset);
    if (rc != GPP_OK) return rc;
    GemmOp co = gemm_default();
    co.A = h->g_U;
    co.lda = (int)h->np;
    co.B = h->iset.U;
    co.ldb = (int)h->np;
    co.C = h->n_C;
    co.ldc = (int)h->iset.mp;
    co.tiles_m = co.tiles_m_last = c.tiles;
    co.tiles_n = iset.tiles;
    co.klo_c = 0;
    co.khi_c = h->T;
    co.alpha = -1.0;
    co.beta = 1.0;
    CK(launch_gemm(co, true, true, 1, h->st));
    QSyrkArgs ga;
    memset(&ga, 0, sizeof(ga));
    ga.U = h->n_C;
    ga.ldu = h->iset.mp;
    ga.kcols = (int)h->i_m;
    ga.q = s.q;
    ga.qpt = s.qpt;
    ga.nb = c.nb;
    ga.cov = h->n_G;
    CK(launch_qbatch_gram(ga, c.tiles, h->st));
    NipvArgs na;
    memset(&na, 0, sizeof(na));
    na.blk = h->q_buf;
    na.gram = h->n_G;
    na.ainv = h->n_Ai;
    na.q = s.q;
    na.nb = c.nb;
    na.inv_m = 1.0 / (double)h->i_m;
    na.vbar = h->i_vbar;
    na.grad = grad ? 1 : 0;
    na.value = h->a_val;
    na.jitter = h->a_jit;
    na.info = h->a_info;
    CK(launch_nipv_block(na, h->st));
    CK(cudaMemcpyAsync(values + c.bt0, h->a_val, sizeof(double) * c.nb, cudaMemcpyDefault, h->st));
    if (jitter) CK(cudaMemcpyAsync(jitter + c.bt0, h->a_jit, sizeof(double) * c.nb, cudaMemcpyDefault, h->st));
    return GPP_OK;
}

// the backward's integration-set terms after W: -C_bar^T = blockdiag(-2 A^-1 / M) C^T in place over C^T, then
// W += C_bar^T V_I, the K* term that reaches U_t through C_t (the finish subtracts W's partials)
static int nipv_w_terms(gpp_handle* h, const QBatchSpec& s, const QChunk& c) {
    // each CTA stages the 32-column panel of its tile in shared memory before it writes that same panel
    QWArgs cw;
    cw.V = h->n_C;
    cw.ldv = h->iset.mp;
    cw.G = h->n_Ai;
    cw.q = s.q;
    cw.qpt = s.qpt;
    cw.nb = c.nb;
    cw.W = h->n_C;
    cw.ldw = h->iset.mp;
    qbatch_w_kernel<<<dim3((unsigned)(h->iset.mp / QB_KC), (unsigned)c.tiles), QB_THREADS, 0, h->st>>>(cw);
    CK(cudaGetLastError());
    count_launch();
    GemmOp wo = gemm_default();
    wo.A = h->n_C;
    wo.lda = (int)h->iset.mp;
    wo.B = h->i_V;
    wo.ldb = (int)h->np;
    wo.C = h->g_U;
    wo.ldc = (int)h->np;
    wo.tiles_m = wo.tiles_m_last = c.tiles;
    wo.tiles_n = h->T;
    wo.klo_c = 0;
    wo.khi_c = (int)(h->iset.mp / CT);
    wo.alpha = -1.0;
    wo.beta = 1.0;
    CK(launch_gemm(wo, true, false, 1, h->st));
    return GPP_OK;
}

extern "C" int gpp_nipv_qbatch(gpp_handle* h, int64_t b, int32_t q, const double* xq, const int32_t* level_idx,
                               const int32_t* noise_idx, double* values, double* d_xq, double* jitter) {
    int rc = check_rows(h, "gpp_nipv_qbatch", qbatch_count_err(b, q), b, xq, level_idx);
    if (rc != GPP_OK) return rc;
    if (!ipv_valid(h)) ARG_FAIL("gpp_nipv_qbatch: no integration set for the current factor (call gpp_ipv_points)");
    if (!values) ARG_FAIL("gpp_nipv_qbatch: values missing");
    if (b == 0) return GPP_OK;
    const QBatchSpec s = qbatch_spec(b, q);
    // the candidates are fantasised with their observation noise (include_noise = 1); the mean is not needed
    const Rows r = {xq, level_idx, noise_idx, nullptr, 1, 0.0};
    const bool grad = d_xq && h->dq > 0;
    // values, jitters and the status word in the acquisition buffers (no base samples); C^T of one chunk, its q x q Gram
    // and A^-1 blocks and, with the gradient, the partials over the T training and the set's column tiles
    if ((rc = qbatch_setup(h, s)) != GPP_OK || (rc = ensure_acq_buffers(h, 0)) != GPP_OK) return rc;
    const long long step = nipv_step(h), imt = h->iset.mp / CT;
    CK(h->n_C.reserve(step * h->iset.mp, h->st));
    CK(h->n_G.reserve(step * q, h->st));
    CK(h->n_Ai.reserve(step * q, h->st));
    CK(h->n_pm.reserve(grad ? step * (h->T + imt) * h->dq : 0, h->st));
    CK(h->n_pv.reserve(grad ? step * (h->T + imt) * h->dq : 0, h->st));
    CK(cudaMemsetAsync(h->a_info, 0, sizeof(int), h->st));
    for (long long base = 0; base < qbatch_rows(s); base += step) {
        const QChunk c = qbatch_chunk(s, base, step);
        if ((rc = qbatch_front(h, s, r, c)) != GPP_OK || (rc = qbatch_sigma(h, s, r, c)) != GPP_OK ||
            (rc = nipv_forward(h, s, c, values, jitter, grad)) != GPP_OK)
            return rc;
        if (grad) {  // A_bar_t is in q_buf already
            const Panels rows = chunk_panels(h, c.mc);
            double* pm_i = h->n_pm + (size_t)h->T * h->dq * step;  // partials over the set's column tiles
            double* pv_i = h->n_pv + (size_t)h->T * h->dq * step;
            if ((rc = v_gemm(h, h->g_U, h->c_K, c.tiles)) != GPP_OK || (rc = qbatch_w(h, s, c)) != GPP_OK ||
                (rc = nipv_w_terms(h, s, c)) != GPP_OK ||
                (rc = grad_tiles(h, rows, training_panels(h), h->alpha, h->g_U, h->np, h->n_pm, h->n_pv, step)) !=
                    GPP_OK ||
                (rc = grad_tiles(h, rows, ipv_panels(h), h->i_zero, h->n_C, h->iset.mp, pm_i, pv_i, step)) != GPP_OK ||
                (rc = qbatch_grad_finish(h, s, c, h->n_pm, h->n_pv, step, h->T + (int)imt, nullptr, d_xq)) != GPP_OK)
                return rc;
        }
        if ((rc = qbatch_status(h, "gpp_nipv_qbatch",
                                "gpp_nipv_qbatch: NaN in a t-batch posterior or its integrated variance")) != GPP_OK)
            return rc;
    }
    return GPP_OK;
}

// ---------------------------------------------------------------------------------------------
// One-shot knowledge gradient (kg.cuh): the gpp_acq_qbatch chunks with every row's observation noise, then per t-batch
// the factor of the actual rows' block, the F fantasy solves and the value in one CTA; with d_xq, the adjoint
// (Sigma_bar_t, mu_bar) feeds the q-batch backward in the same chunk, which gives d_xq of the fantasy rows too.
extern "C" int gpp_kg_qbatch(gpp_handle* h, int64_t b, int32_t q, int32_t n_fantasies, const double* xq,
                             const int32_t* level_idx, const int32_t* noise_idx, const int32_t* mean_idx, int maximize,
                             const double* base_samples, double* values, double* d_xq, double* jitter) {
    const char* bad = nullptr;
    if (q < 1 || n_fantasies < 1) bad = "q and n_fantasies must be >= 1";
    else if ((long long)q + n_fantasies > GPP_MAX_QBATCH) bad = "q + n_fantasies must be <= GPP_MAX_QBATCH";
    else if (b < 0) bad = "b must be >= 0";
    int rc = check_rows(h, "gpp_kg_qbatch", bad, b, xq, level_idx);
    if (rc != GPP_OK) return rc;
    if (!base_samples || !values) ARG_FAIL("gpp_kg_qbatch: base_samples / values missing");
    if (b == 0) return GPP_OK;
    const int q_tot = q + n_fantasies;
    const QBatchSpec s = qbatch_spec(b, q_tot);
    // the actual rows are fantasised with their observation noise (include_noise = 1, NULL noise_idx: group 0)
    const Rows r = {xq, level_idx, noise_idx, mean_idx, 1, 0.0};
    const bool grad = d_xq && h->dq > 0;
    const long long e_elems = (long long)n_fantasies * q;
    if ((rc = qbatch_setup(h, s)) != GPP_OK || (rc = ensure_acq_buffers(h, e_elems)) != GPP_OK) return rc;
    CK(cudaMemcpyAsync(h->a_E, base_samples, sizeof(double) * e_elems, cudaMemcpyDefault, h->st));
    CK(cudaMemsetAsync(h->a_info, 0, sizeof(int), h->st));
    KgArgs ka;
    memset(&ka, 0, sizeof(ka));
    ka.blk = h->q_buf;
    ka.mu = h->c_mu;
    ka.gm = h->q_gm;
    ka.E = h->a_E;
    ka.q = q;
    ka.nf = n_fantasies;
    ka.qpt = s.qpt;
    ka.sgn = maximize ? 1.0 : -1.0;
    ka.grad = grad ? 1 : 0;
    ka.value = h->a_val;
    ka.jitter = h->a_jit;
    ka.info = h->a_info;
    const long long step = h->g_step;
    for (long long base = 0; base < qbatch_rows(s); base += step) {
        const QChunk c = qbatch_chunk(s, base, step);
        if ((rc = qbatch_front(h, s, r, c)) != GPP_OK || (rc = qbatch_sigma(h, s, r, c)) != GPP_OK) return rc;
        if (grad) CK(cudaMemsetAsync(h->q_gm, 0, sizeof(double) * c.mcp, h->st));
        ka.nb = c.nb;
        CK(launch_kg_block(ka, h->st));
        CK(cudaMemcpyAsync(values + c.bt0, h->a_val, sizeof(double) * c.nb, cudaMemcpyDefault, h->st));
        if (jitter) CK(cudaMemcpyAsync(jitter + c.bt0, h->a_jit, sizeof(double) * c.nb, cudaMemcpyDefault, h->st));
        if (grad) {  // Sigma_bar_t is in q_buf and mu_bar in q_gm already
            if ((rc = v_gemm(h, h->g_U, h->c_K, c.tiles)) != GPP_OK || (rc = qbatch_w(h, s, c)) != GPP_OK) return rc;
            if ((rc = grad_tiles(h, chunk_panels(h, c.mc), training_panels(h), h->alpha, h->g_U, h->np, h->g_part_m,
                                 h->g_part_v, step)) != GPP_OK)
                return rc;
            if ((rc = qbatch_grad_finish(h, s, c, h->g_part_m, h->g_part_v, step, h->T, h->q_gm, d_xq)) != GPP_OK)
                return rc;
        }
        if ((rc = qbatch_status(h, "gpp_kg_qbatch",
                                "gpp_kg_qbatch: NaN in a t-batch posterior or its fantasy means")) != GPP_OK)
            return rc;
    }
    return GPP_OK;
}

// ---------------------------------------------------------------------------------------------
// GIBBON (gibbon.cuh): the gpp_acq_qbatch chunks with the latent block (no noise), then per t-batch the noise of the
// actual rows, the factor of their block, the diversity and quality terms and the value in one CTA; with d_xq, the
// adjoint (Sigma_bar_t, mu_bar) feeds the q-batch backward in the same chunk, which gives d_xq of the target rows too.
extern "C" int gpp_gibbon_qbatch(gpp_handle* h, int64_t b, int32_t q, int32_t projected, const double* xq,
                                 const int32_t* level_idx, const int32_t* noise_idx, const int32_t* mean_idx,
                                 int maximize, int64_t n_max_values, const double* max_values, double* values,
                                 double* d_xq, double* jitter) {
    const char* bad = nullptr;
    if (q < 1) bad = "q must be >= 1";
    else if (projected != 0 && projected != 1) bad = "projected must be 0 or 1";
    else if ((long long)q * (1 + projected) > GPP_MAX_QBATCH) bad = "q * (1 + projected) must be <= GPP_MAX_QBATCH";
    else if (b < 0) bad = "b must be >= 0";
    int rc = check_rows(h, "gpp_gibbon_qbatch", bad, b, xq, level_idx);
    if (rc != GPP_OK) return rc;
    if (n_max_values < 1 || n_max_values > GPP_MAX_MC_SAMPLES)
        ARG_FAIL("gpp_gibbon_qbatch: n_max_values must be in [1, GPP_MAX_MC_SAMPLES]");
    if (!max_values || !values) ARG_FAIL("gpp_gibbon_qbatch: max_values / values missing");
    if (b == 0) return GPP_OK;
    const int q_tot = q * (1 + projected);
    const QBatchSpec s = qbatch_spec(b, q_tot);
    // the latent block: the actual rows' noise is added inside gibbon_block_kernel, the target rows stay noiseless
    const Rows r = {xq, level_idx, noise_idx, mean_idx, 0, 0.0};
    const bool grad = d_xq && h->dq > 0;
    if ((rc = qbatch_setup(h, s)) != GPP_OK || (rc = ensure_acq_buffers(h, n_max_values)) != GPP_OK) return rc;
    CK(cudaMemcpyAsync(h->a_E, max_values, sizeof(double) * n_max_values, cudaMemcpyDefault, h->st));
    CK(cudaMemsetAsync(h->a_info, 0, sizeof(int), h->st));
    GibbonArgs ga;
    memset(&ga, 0, sizeof(ga));
    ga.blk = h->q_buf;
    ga.mu = h->c_mu;
    ga.gm = h->q_gm;
    ga.noise_idx = noise_idx ? h->c_noise.p : nullptr;
    ga.noise = hyp_noise(h);
    ga.n_noise = h->n_noise;
    ga.mv = h->a_E;
    ga.K = (int)n_max_values;
    ga.q = q;
    ga.q_tot = q_tot;
    ga.qpt = s.qpt;
    ga.sgn = maximize ? 1.0 : -1.0;
    ga.grad = grad ? 1 : 0;
    ga.value = h->a_val;
    ga.jitter = h->a_jit;
    ga.info = h->a_info;
    const long long step = h->g_step;
    for (long long base = 0; base < qbatch_rows(s); base += step) {
        const QChunk c = qbatch_chunk(s, base, step);
        if ((rc = qbatch_front(h, s, r, c)) != GPP_OK || (rc = qbatch_sigma(h, s, r, c)) != GPP_OK) return rc;
        if (grad) CK(cudaMemsetAsync(h->q_gm, 0, sizeof(double) * c.mcp, h->st));
        ga.nb = c.nb;
        CK(launch_gibbon_block(ga, h->st));
        CK(cudaMemcpyAsync(values + c.bt0, h->a_val, sizeof(double) * c.nb, cudaMemcpyDefault, h->st));
        if (jitter) CK(cudaMemcpyAsync(jitter + c.bt0, h->a_jit, sizeof(double) * c.nb, cudaMemcpyDefault, h->st));
        if (grad) {  // Sigma_bar_t is in q_buf and mu_bar in q_gm already
            if ((rc = v_gemm(h, h->g_U, h->c_K, c.tiles)) != GPP_OK || (rc = qbatch_w(h, s, c)) != GPP_OK) return rc;
            if ((rc = grad_tiles(h, chunk_panels(h, c.mc), training_panels(h), h->alpha, h->g_U, h->np, h->g_part_m,
                                 h->g_part_v, step)) != GPP_OK)
                return rc;
            if ((rc = qbatch_grad_finish(h, s, c, h->g_part_m, h->g_part_v, step, h->T, h->q_gm, d_xq)) != GPP_OK)
                return rc;
        }
        if ((rc = qbatch_status(h, "gpp_gibbon_qbatch",
                                "gpp_gibbon_qbatch: NaN in a t-batch posterior or its GIBBON value")) != GPP_OK)
            return rc;
    }
    return GPP_OK;
}

// Max-value quartiles (gibbon.cuh): the marginals by the pointwise family into v_mu / v_var (bitwise gpp_predict's at
// include_noise = 0, min_var = 1e-8), the bracket, its widening (one host check per step) and 40 bisection steps of
// the three brackets on the device
extern "C" int gpp_max_value_quartiles(gpp_handle* h, int64_t m, const double* xq, const int32_t* level_idx,
                                       const int32_t* mean_idx, int maximize, double* quartiles) {
    int rc = check_rows(h, "gpp_max_value_quartiles", m < 1 ? "m must be >= 1" : nullptr, m, xq, level_idx);
    if (rc != GPP_OK) return rc;
    if (!quartiles) ARG_FAIL("gpp_max_value_quartiles: quartiles missing");
    CK(cudaSetDevice(h->device));
    const int nblk = mv_blocks(m);
    CK(h->v_mu.reserve(m, h->st));
    CK(h->v_var.reserve(m, h->st));
    CK(h->v_part.reserve((size_t)nblk * 4, h->st));
    CK(h->v_state.reserve(MV_STATE, h->st));
    CK(h->v_nan.reserve(1, h->st));
    const Rows r = {xq, level_idx, nullptr, mean_idx, 0, 1e-8};
    if ((rc = predict_rows(h, m, r, h->v_mu, h->v_var, nullptr, nullptr, nullptr)) != GPP_OK) return rc;
    const double sgn = maximize ? 1.0 : -1.0;
    mv_range_kernel<<<nblk, MV_THREADS, 0, h->st>>>(h->v_mu, h->v_var, m, sgn, h->v_part);
    CK(cudaGetLastError());
    mv_range_finish_kernel<<<1, 32, 0, h->st>>>(h->v_part, nblk, h->v_state, h->v_nan);
    CK(cudaGetLastError());
    count_launch();
    count_launch();
    int nan = 0;
    CK(cudaMemcpyAsync(&nan, h->v_nan, sizeof(int), cudaMemcpyDeviceToHost, h->st));
    CK(cudaStreamSynchronize(h->st));
    if (nan) {
        g_err = "gpp_max_value_quartiles: NaN or infinity in a candidate's posterior mean or variance";
        return GPP_ERR_NAN;
    }
    auto step = [&](int widen) -> cudaError_t {
        mv_loglik_kernel<<<nblk, MV_THREADS, 0, h->st>>>(h->v_mu, h->v_var, m, sgn, h->v_state, widen ? 1 : MV_PTS,
                                                         h->v_part);
        mv_step_kernel<<<1, 32, 0, h->st>>>(h->v_part, nblk, h->v_state, widen);
        count_launch();
        count_launch();
        return cudaGetLastError();
    };
    // widen hi until l(hi) >= log 3/4: for m >~ 1e6 the first bracket misses the upper quartile.  With finite marginals
    // one doubling puts every term at z >= 15, where log Phi(15) = -3.7e-51, so a second check always passes; the
    // bound only keeps the loop finite.
    for (int it = 0;; it++) {
        if (it == 8) {
            g_err = "gpp_max_value_quartiles: l(hi) stays below log 3/4 after 8 doublings of the bracket";
            return GPP_ERR_NAN;
        }
        CK(step(1));
        double flag = 0.0;
        CK(cudaMemcpyAsync(&flag, h->v_state.p + 11, sizeof(double), cudaMemcpyDeviceToHost, h->st));
        CK(cudaStreamSynchronize(h->st));
        if (flag == 0.0) break;
    }
    // 40 halvings leave each quartile within 2^-41 (hi - lo) < 1e-12 (hi - lo) of the midpoint returned
    for (int it = 0; it < 40; it++) CK(step(0));
    double state[MV_STATE];
    CK(cudaMemcpyAsync(state, h->v_state, sizeof(double) * MV_STATE, cudaMemcpyDeviceToHost, h->st));
    CK(cudaStreamSynchronize(h->st));
    for (int p = 0; p < MV_PTS; p++) {
        if (!std::isfinite(state[8 + p])) {
            g_err = "gpp_max_value_quartiles: a quartile is not finite";
            return GPP_ERR_NAN;
        }
    }
    CK(cudaMemcpyAsync(quartiles, h->v_state.p + 8, sizeof(double) * MV_PTS, cudaMemcpyDefault, h->st));
    CK(cudaStreamSynchronize(h->st));
    return GPP_OK;
}

// ---------------------------------------------------------------------------------------------
extern "C" int gpp_probe_dgemm(int device, int m, int n, int k, int iters, float* ms_out) {
    if (m <= 0 || n <= 0 || k <= 0 || (m % 128) || (n % 128) || (k % 128) || iters <= 0 || !ms_out)
        ARG_FAIL("gpp_probe_dgemm: sizes must be positive multiples of 128");
    CK(cudaSetDevice(device));
    CK(gemm_set_attributes());
    double *A = nullptr, *B = nullptr, *C = nullptr;
    CK(dev_alloc(&A, (size_t)m * k));
    CK(dev_alloc(&B, (size_t)n * k));
    CK(dev_alloc(&C, (size_t)m * n));
    {
        // random operands in [-1, 1): power draw (and therefore clocks) of the DMMA pipe depends on the data
        std::vector<double> hA((size_t)m * k), hB((size_t)n * k);
        unsigned long long sd = 0x9E3779B97F4A7C15ull;
        auto rnd = [&]() {
            sd ^= sd << 13; sd ^= sd >> 7; sd ^= sd << 17;
            return (double)(sd >> 11) * (2.0 / 9007199254740992.0) - 1.0;
        };
        for (auto& v : hA) v = rnd();
        for (auto& v : hB) v = rnd();
        CK(cudaMemcpy(A, hA.data(), sizeof(double) * m * k, cudaMemcpyHostToDevice));
        CK(cudaMemcpy(B, hB.data(), sizeof(double) * n * k, cudaMemcpyHostToDevice));
    }
    GemmOp op = gemm_default();
    op.A = A;
    op.lda = k;
    op.B = B;
    op.ldb = k;
    op.C = C;
    op.ldc = n;
    op.tiles_m = op.tiles_m_last = m / 128;
    op.tiles_n = n / 128;
    op.klo_c = 0;
    op.khi_c = k / 128;
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0));
    CK(cudaEventCreate(&e1));
    for (int i = 0; i < 2; i++) CK(launch_gemm(op, true, true, 1, 0));
    CK(cudaEventRecord(e0, 0));
    for (int i = 0; i < iters; i++) CK(launch_gemm(op, true, true, 1, 0));
    CK(cudaEventRecord(e1, 0));
    CK(cudaEventSynchronize(e1));
    float ms = 0.f;
    CK(cudaEventElapsedTime(&ms, e0, e1));
    *ms_out = ms / iters;
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(A);
    cudaFree(B);
    cudaFree(C);
    return GPP_OK;
}

extern "C" int gpp_probe_i8(int device, int n_cols, int iters, double* tops_out) {
    if (!tops_out || iters <= 0 || (n_cols != 64 && n_cols != 128 && n_cols != 256)) ARG_FAIL("gpp_probe_i8: bad arguments");
    CK(cudaSetDevice(device));
    iters = (iters + 7) / 8 * 8;
    if (n_cols == 64) CK(oz_probe_rate_n<64>(iters, tops_out));
    else if (n_cols == 128) CK(oz_probe_rate_n<128>(iters, tops_out));
    else CK(oz_probe_rate_n<256>(iters, tops_out));
    return GPP_OK;
}
