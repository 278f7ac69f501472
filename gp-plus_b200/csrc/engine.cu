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
#include "objective.h"
#include "predict.cuh"
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
// GPP_FP64) and the development switches, per handle and process-wide (int fields only: compared with memcmp).
// A parked handle is handed back only when the configuration in force now equals the one it was built under.
struct CreateConfig {
    int lookahead, graph, early_out, small_block;                                    // per handle
    int panel_blocks, overlap_inverse, gemm_bm, gemm_stagger, oz_items_per_cta;       // process globals
    int int8;                                                                         // INT8-sliced O(N^3) stages
    int oz_min_trail, oz_min_level, oz_next, oz_inner, oz_lazy, oz_kinv_levels, oz_lazy_min, oz_lazy_pb, oz_stagger;
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
    // prediction chunk buffers
    long long mc_alloc = 0;
    double *c_xq = nullptr, *c_xs = nullptr, *c_nrm = nullptr, *c_zpt = nullptr, *c_K = nullptr;
    int *c_lvl = nullptr, *c_noise = nullptr, *c_mean = nullptr, *c_cost = nullptr;
    double *c_mean_part = nullptr, *c_rowsq = nullptr, *c_mu = nullptr, *c_var = nullptr, *c_score = nullptr;
    double* c_blk_best = nullptr;
    long long* c_blk_idx = nullptr;
    double* acq_par = nullptr;  // [cost n_cost | best_f n_cost]
    int* acq_kind = nullptr;
    int acq_cap = 0;
    bool factorized = false;
    double last_jitter = 0.0;
    cudaEvent_t ev[EV_COUNT];
    bool ev_valid[EV_COUNT];
    gpp_timings tm;
    CholLookahead la;
    bool use_lookahead = true;
    int small_block = 0;     // T <= 16: CTAs of the one-launch factorisation (GPP_SMALL_BLOCK; 0 = launch chain)
    OzCtx* oz = nullptr;     // INT8-sliced tcgen05 path of the O(N^3) stages (large problems; GPP_FP64=dmma turns it off)
    // CUDA-graph replay of one whole evaluation (small problems are launch-bound): [want_grad]
    cudaGraphExec_t graph_exec[2] = {nullptr, nullptr};
    long long graph_kernels[2] = {0, 0};
    bool use_graph = false;
    bool early_out = true;   // read the factorisation status before enqueueing the rest (non-graph path)
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

extern "C" int gpp_version(void) { return 106; }

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

template <typename Tp>
static cudaError_t dev_alloc(Tp** p, size_t count) {
    return cudaMalloc((void**)p, std::max<size_t>(count, 1) * sizeof(Tp));
}

static void destroy_now(gpp_handle* h) {
    if (!h) return;
    cudaSetDevice(h->device);
    if (h->st) cudaStreamSynchronize(h->st);
    void* dptrs[] = {h->slab, h->c_xq, h->c_xs, h->c_nrm, h->c_zpt, h->c_K, h->c_lvl,
                     h->c_noise, h->c_mean, h->c_cost, h->c_mean_part, h->c_rowsq, h->c_mu, h->c_var, h->c_score,
                     h->c_blk_best, h->c_blk_idx, h->acq_par, h->acq_kind};
    for (void* p : dptrs)
        if (p) cudaFree(p);
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

// the configuration a handle with T tile rows gets when it is created now (defaults are the production configuration;
// the process globals keep the value an earlier gpp_create gave them unless the environment sets them again)
static CreateConfig read_config(int T) {
    CreateConfig c;
    memset(&c, 0, sizeof(c));
    const char* e;
    c.lookahead = 1;
    if ((e = getenv("GPP_CHOL")) != nullptr) c.lookahead = strcmp(e, "blocked") != 0;
    c.graph = T <= 16;  // N <= 2048: an evaluation is a chain of ~25-100 tiny launches
    if ((e = getenv("GPP_GRAPH")) != nullptr) c.graph = atoi(e) != 0;
    c.early_out = 1;
    if ((e = getenv("GPP_EARLY_OUT")) != nullptr) c.early_out = atoi(e) != 0;
    c.small_block = 0;
    if ((e = getenv("GPP_SMALL_BLOCK")) != nullptr) c.small_block = atoi(e);
    c.panel_blocks = g_panel_blocks;
    if ((e = getenv("GPP_PANEL")) != nullptr) c.panel_blocks = atoi(e);
    c.overlap_inverse = g_overlap_inverse;
    if ((e = getenv("GPP_OVERLAP_INV")) != nullptr) c.overlap_inverse = atoi(e);
    c.gemm_bm = g_gemm_bm;
    if ((e = getenv("GPP_GEMM_BM")) != nullptr) c.gemm_bm = atoi(e) == 64 ? 64 : 128;
    c.gemm_stagger = g_gemm_stagger;
    if ((e = getenv("GPP_STAGGER")) != nullptr) c.gemm_stagger = atoi(e);
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
    c.oz_items_per_cta = g_oz_items_per_cta;
    OzCtx d;   // defaults only (init() allocates)
    c.oz_min_trail = d.min_trailing_tiles;
    c.oz_min_level = d.min_level_tiles;
    c.oz_next = d.next_on_oz;
    c.oz_inner = d.inner_min_k;
    c.oz_lazy = d.lazy;
    c.oz_kinv_levels = d.kinv_levels;
    c.oz_lazy_min = d.lazy_min_tiles;
    c.oz_lazy_pb = d.lazy_pb;
    c.oz_stagger = d.stagger;
    if (c.int8) {
        if ((e = getenv("GPP_OZ_IPC")) != nullptr) c.oz_items_per_cta = atoi(e) > 0 ? atoi(e) : 2;
        if ((e = getenv("GPP_OZ_MIN_TRAIL")) != nullptr) c.oz_min_trail = atoi(e);
        if ((e = getenv("GPP_OZ_MIN_LEVEL")) != nullptr) c.oz_min_level = atoi(e);
        if ((e = getenv("GPP_OZ_NEXT")) != nullptr) c.oz_next = atoi(e);
        if ((e = getenv("GPP_OZ_INNER")) != nullptr) c.oz_inner = atoi(e);
        if ((e = getenv("GPP_OZ_LAZY")) != nullptr) c.oz_lazy = atoi(e);
        if ((e = getenv("GPP_OZ_KINV_LEVELS")) != nullptr) c.oz_kinv_levels = atoi(e);
        if ((e = getenv("GPP_OZ_LAZY_MIN")) != nullptr) c.oz_lazy_min = atoi(e);
        if ((e = getenv("GPP_OZ_LAZY_PB")) != nullptr) c.oz_lazy_pb = std::min(std::max(atoi(e), 2), OzCtx::LAZY_PB);
        if ((e = getenv("GPP_OZ_STAGGER")) != nullptr) c.oz_stagger = atoi(e);
    }
    return c;
}

static void apply_globals(const CreateConfig& c) {
    g_panel_blocks = c.panel_blocks;
    g_overlap_inverse = c.overlap_inverse;
    g_gemm_bm = c.gemm_bm;
    g_gemm_stagger = c.gemm_stagger;
    g_oz_items_per_cta = c.oz_items_per_cta;
}

// per-handle switches (h->oz, when the handle has one, must exist already)
static void apply_handle_config(gpp_handle* h, const CreateConfig& c) {
    h->cfg = c;
    h->use_lookahead = c.lookahead != 0;
    h->use_graph = c.graph != 0;
    h->early_out = c.early_out != 0;
    h->small_block = c.small_block;
    if (h->oz) {
        h->oz->min_trailing_tiles = c.oz_min_trail;
        h->oz->min_level_tiles = c.oz_min_level;
        h->oz->next_on_oz = c.oz_next;
        h->oz->inner_min_k = c.oz_inner;
        h->oz->lazy = c.oz_lazy;
        h->oz->kinv_levels = c.oz_kinv_levels;
        h->oz->lazy_min_tiles = c.oz_lazy_min;
        h->oz->lazy_pb = c.oz_lazy_pb;
        h->oz->stagger = c.oz_stagger;
    }
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
    if (pooling && h->slab_bytes <= kPoolMaxHandleBytes && h->mc_alloc == 0) {
        cudaSetDevice(h->device);
        if (h->st) cudaStreamSynchronize(h->st);
        std::lock_guard<std::mutex> lk(g_pool_mu);
        if (g_pool.size() < kPoolMaxHandles && g_pool_bytes + h->slab_bytes <= kPoolMaxBytes) {
            h->layout.set = false;
            h->factorized = false;
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
    apply_globals(cfg);
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
            apply_handle_config(reuse, cfg);   // (a failed graph capture may have switched the replay off)
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
    CKH(h->la.init(h->T));
    if (cfg.int8) {
        h->oz = new OzCtx();
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
    apply_handle_config(h, cfg);

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

// upload the staged hyper-parameters and prepare the per-point panels of the training set
static int stage_prep(gpp_handle* h) {
    CK(cudaMemcpyAsync(h->hyp, h->hyp_host, sizeof(double) * h->hyp_len, cudaMemcpyHostToDevice, h->st));
    PrepArgs pa;
    pa.xq = h->xq;
    pa.level_idx = h->level_idx;
    pa.w = hyp_w(h);
    pa.centre = h->centre;
    pa.ztab = hyp_z(h);
    pa.n = (int)h->n;
    pa.np = (int)h->np;
    pa.dq = h->dq;
    pa.dqp = h->dqp;
    pa.dz = h->dz;
    pa.n_combo = h->n_combo;
    pa.n_pass = h->n_pass;
    pa.xs = h->xs;
    pa.xst = h->xst;
    pa.nrm = h->nrm;
    pa.zpt = h->zpt;
    const int nb = (int)((h->np + 255) / 256);
    prep_points_kernel<<<nb, 256, 0, h->st>>>(pa);
    CK(cudaGetLastError());
    count_launch();
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
    ca.xs_r = ca.xs_c = h->xs;
    ca.nrm_r = ca.nrm_c = h->nrm;
    ca.out = h->A;
    ca.ld = h->np;
    ca.n_r = ca.n_c = (int)h->n;
    ca.tiles_r = ca.tiles_c = h->T;
    ca.tri = 1;
    ca.same = 1;
    ca.pad_identity = 1;
    ca.dqp = h->dqp;
    ca.dz = h->dz;
    ca.sf2 = h->sf2;
    ca.sf2_dev = hyp_sf2(h);
    ca.diag_add = h->diag_add;
    ca.scale = 1.0 / (double)h->n_pass;
    for (int p = 0; p < h->n_pass; p++) {  // K = (1/k) sum_p K_p: one launch per latent table
        ca.zpt_r = ca.zpt_c = h->zpt + (size_t)p * h->np * ZP;
        ca.accum = p > 0;
        ca.last = p == h->n_pass - 1;
        CK(launch_cov(ca, h->kernel, h->st));
    }
    mark(h, EV_COV);
    if (h->small_block > 0 && h->T <= 16) {
        // small problems: the whole factorisation is one dataflow launch (block_potrf_kernel) instead of a chain of
        // T leaf / TRSM / update launches.  Inside a captured graph the launch arguments are frozen, so the tile flags
        // are cleared by a memset node and the epoch is constant.
        CK(cudaMemsetAsync(h->la.blk_flags, 0, 256 * sizeof(int), h->st));
        CK(launch_block_potrf(h->A, h->M, (int)h->np, 0, h->T, h->logdet_part, h->info, h->la.blk_flags, 1, h->small_block,
                              h->st));
    } else if (h->use_lookahead && h->oz && h->oz->ready && h->oz->lazy && h->T >= h->oz->lazy_min_tiles)
        CK(potrf_lazy(h->A, h->M, (int)h->np, h->T, h->logdet_part, h->info, h->st, h->la, h->S, *h->oz));
    else if (h->use_lookahead)
        CK(potrf_lookahead(h->A, h->M, (int)h->np, h->T, h->logdet_part, h->info, h->st, h->la, h->S, h->oz));
    else
        CK(potrf_blocked(h->A, h->M, (int)h->np, h->T, h->logdet_part, h->info, h->st));
    mark(h, EV_CHOL);
    return GPP_OK;
}

// M <- L^-1, v = M r, alpha = M^T v
static int stage_inverse_solve(gpp_handle* h) {
    if (h->use_lookahead && h->la.inv_pending) {
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
        if (h->use_lookahead && h->la.inv_pending) {
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
        } else if (h->early_out) {
            int failed = 0;
            int rc = enqueue_eval_early_out(h, want_grad, &failed);
            if (rc != GPP_OK) return rc;
            mark(h, EV_END);
            CK(cudaStreamSynchronize(h->st));
            if (h->la.timeline) h->la.dump_timeline(h->oz ? (h->T + h->oz->lazy_pb - 1) / h->oz->lazy_pb : h->la.panels);
            info = failed ? failed : (int)h->res_host[2];
        } else {
            int rc = enqueue_eval(h, want_grad);
            if (rc != GPP_OK) return rc;
            mark(h, EV_END);
            CK(cudaStreamSynchronize(h->st));
            info = (int)h->res_host[2];
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
    h->pending = false;
    rc = run_eval(h, hy, want_grad ? 1 : 0);
    if (rc != GPP_OK) return rc;
    h->factorized = true;
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
    h->pending = false;
    int rc = run_eval(h, &hy, want_grad ? 1 : 0);
    if (rc != GPP_OK) return rc;
    h->factorized = true;
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
    fill_hyper_host(h, hy, 0.0);
    if ((rc = stage_prep(h)) != GPP_OK) return rc;
    CovArgs ca;
    memset(&ca, 0, sizeof(ca));
    ca.xs_r = ca.xs_c = h->xs;
    ca.nrm_r = ca.nrm_c = h->nrm;
    ca.out = h->S;
    ca.ld = h->np;
    ca.n_r = ca.n_c = (int)h->n;
    ca.tiles_r = ca.tiles_c = h->T;
    ca.tri = 0;
    ca.same = 1;
    ca.pad_identity = 0;
    ca.dqp = h->dqp;
    ca.dz = h->dz;
    ca.sf2 = h->sf2;
    ca.scale = 1.0 / (double)h->n_pass;
    for (int p = 0; p < h->n_pass; p++) {
        ca.zpt_r = ca.zpt_c = h->zpt + (size_t)p * h->np * ZP;
        ca.accum = p > 0;
        ca.last = p == h->n_pass - 1;
        CK(launch_cov(ca, h->kernel, h->st));
    }
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
    rc = run_eval(h, hy, 0);
    if (rc != GPP_OK) return rc;
    h->factorized = true;
    return GPP_OK;
}

// ---------------------------------------------------------------------------------------------
static int ensure_chunk_buffers(gpp_handle* h, long long m) {
    // K* chunk of at most 2^27 doubles (1 GiB)
    long long cap = ((1LL << 27) / h->np) / 128 * 128;
    if (cap < 128) cap = 128;
    long long want = std::min((m + 127) / 128 * 128, cap);
    if (want <= h->mc_alloc) return GPP_OK;
    void* olds[] = {h->c_xq, h->c_xs, h->c_nrm, h->c_zpt, h->c_K, h->c_lvl, h->c_noise, h->c_mean, h->c_cost,
                    h->c_mean_part, h->c_rowsq, h->c_mu, h->c_var, h->c_score, h->c_blk_best, h->c_blk_idx};
    for (void* p : olds)
        if (p) cudaFree(p);
    h->c_xq = h->c_xs = h->c_nrm = h->c_zpt = h->c_K = nullptr;
    h->c_lvl = h->c_noise = h->c_mean = h->c_cost = nullptr;
    h->c_mean_part = h->c_rowsq = h->c_mu = h->c_var = h->c_score = h->c_blk_best = nullptr;
    h->c_blk_idx = nullptr;
    h->mc_alloc = 0;
    const size_t mc = (size_t)want;
    CK(dev_alloc(&h->c_xq, mc * std::max(h->dq, 1)));
    CK(dev_alloc(&h->c_xs, mc * h->dqp));
    CK(dev_alloc(&h->c_nrm, mc));
    CK(dev_alloc(&h->c_zpt, mc * ZP * h->n_pass));
    CK(dev_alloc(&h->c_K, mc * (size_t)h->np));
    CK(dev_alloc(&h->c_lvl, mc));
    CK(dev_alloc(&h->c_noise, mc));
    CK(dev_alloc(&h->c_mean, mc));
    CK(dev_alloc(&h->c_cost, mc));
    CK(dev_alloc(&h->c_mean_part, mc * (size_t)h->T));
    CK(dev_alloc(&h->c_rowsq, mc * (size_t)h->T));
    CK(dev_alloc(&h->c_mu, mc));
    CK(dev_alloc(&h->c_var, mc));
    CK(dev_alloc(&h->c_score, mc));
    CK(dev_alloc(&h->c_blk_best, mc / 256 + 1));
    CK(dev_alloc(&h->c_blk_idx, mc / 256 + 1));
    h->mc_alloc = want;
    return GPP_OK;
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

static int predict_impl(gpp_handle* h, long long m, const double* xq, const int32_t* level_idx,
                        const int32_t* noise_idx, const int32_t* mean_idx, int include_noise, double min_var,
                        double* mean, double* var, AcqSpec* acq) {
    if (!h->factorized) ARG_FAIL("predict: call gpp_factorize (or gpp_mll_grad) first");
    if (m <= 0) return GPP_OK;
    if (h->dq > 0 && !xq) ARG_FAIL("predict: xq missing");
    if (h->dz > 0 && !level_idx) ARG_FAIL("predict: level_idx missing");
    CK(cudaSetDevice(h->device));
    int rc = ensure_chunk_buffers(h, m);
    if (rc != GPP_OK) return rc;
    if (acq) {
        if (acq->n_cost <= 0 || !acq->cost || !acq->kind_by_cost || !acq->best_f) ARG_FAIL("acq: cost tables missing");
        if (acq->n_cost > h->acq_cap) {
            if (h->acq_par) cudaFree(h->acq_par);
            if (h->acq_kind) cudaFree(h->acq_kind);
            h->acq_par = nullptr;
            h->acq_kind = nullptr;
            CK(dev_alloc(&h->acq_par, (size_t)2 * acq->n_cost));
            CK(dev_alloc(&h->acq_kind, (size_t)acq->n_cost));
            h->acq_cap = acq->n_cost;
        }
        CK(cudaMemcpyAsync(h->acq_par, acq->cost, sizeof(double) * acq->n_cost, cudaMemcpyDefault, h->st));
        CK(cudaMemcpyAsync(h->acq_par + acq->n_cost, acq->best_f, sizeof(double) * acq->n_cost, cudaMemcpyDefault,
                           h->st));
        CK(cudaMemcpyAsync(h->acq_kind, acq->kind_by_cost, sizeof(int) * acq->n_cost, cudaMemcpyDefault, h->st));
    }
    std::vector<double> hb;
    std::vector<long long> hi;
    const long long MC = h->mc_alloc;
    for (long long base = 0; base < m; base += MC) {
        const long long mc = std::min(MC, m - base);
        const long long mcp = (mc + 127) / 128 * 128;
        const int tiles_r = (int)(mcp / 128);
        if (h->dq > 0)
            CK(cudaMemcpyAsync(h->c_xq, xq + base * h->dq, sizeof(double) * mc * h->dq, cudaMemcpyDefault, h->st));
        if (h->dz > 0)
            CK(cudaMemcpyAsync(h->c_lvl, level_idx + base, sizeof(int) * mc, cudaMemcpyDefault, h->st));
        if (noise_idx) CK(cudaMemcpyAsync(h->c_noise, noise_idx + base, sizeof(int) * mc, cudaMemcpyDefault, h->st));
        if (mean_idx) CK(cudaMemcpyAsync(h->c_mean, mean_idx + base, sizeof(int) * mc, cudaMemcpyDefault, h->st));
        if (acq && acq->cost_idx)
            CK(cudaMemcpyAsync(h->c_cost, acq->cost_idx + base, sizeof(int) * mc, cudaMemcpyDefault, h->st));
        PrepArgs pa;
        pa.xq = h->c_xq;
        pa.level_idx = h->dz > 0 ? h->c_lvl : nullptr;
        pa.w = hyp_w(h);
        pa.centre = h->centre;
        pa.ztab = hyp_z(h);
        pa.n = (int)mc;
        pa.np = (int)mcp;
        pa.dq = h->dq;
        pa.dqp = h->dqp;
        pa.dz = h->dz;
        pa.n_combo = h->n_combo;
        pa.n_pass = h->n_pass;
        pa.xs = h->c_xs;
        pa.xst = nullptr;
        pa.nrm = h->c_nrm;
        pa.zpt = h->c_zpt;
        prep_points_kernel<<<(int)((mcp + 255) / 256), 256, 0, h->st>>>(pa);
        CK(cudaGetLastError());
    count_launch();

        CovArgs ca;
        memset(&ca, 0, sizeof(ca));
        ca.xs_r = h->c_xs;
        ca.nrm_r = h->c_nrm;
        ca.xs_c = h->xs;
        ca.nrm_c = h->nrm;
        ca.out = h->c_K;
        ca.ld = h->np;
        ca.n_r = (int)mc;
        ca.n_c = (int)h->n;
        ca.tiles_r = tiles_r;
        ca.tiles_c = h->T;
        ca.dqp = h->dqp;
        ca.dz = h->dz;
        ca.sf2 = h->sf2;
        ca.alpha = h->alpha;
        ca.mean_part = h->c_mean_part;
        ca.ld_part = MC;
        ca.scale = 1.0 / (double)h->n_pass;
        for (int p = 0; p < h->n_pass; p++) {
            ca.zpt_r = h->c_zpt + (size_t)p * mcp * ZP;
            ca.zpt_c = h->zpt + (size_t)p * h->np * ZP;
            ca.accum = p > 0;
            ca.last = p == h->n_pass - 1;
            CK(launch_cov(ca, h->kernel, h->st));
        }

        GemmOp op = gemm_default();  // V = K* L^-T, only its row sums of squares are kept
        op.A = h->c_K;
        op.lda = (int)h->np;
        op.B = h->M;
        op.ldb = (int)h->np;
        op.C = nullptr;
        op.ldc = 0;
        op.tiles_m = op.tiles_m_last = tiles_r;
        op.tiles_n = h->T;
        op.klo_c = 0;
        op.khi_sel = KSEL_TJ;
        op.khi_c = 1;
        op.epilogue = EPI_ROWSQ;
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
        fa.mean_idx = mean_idx ? h->c_mean : nullptr;
        fa.beta = hyp_beta(h);
        fa.n_mean = h->n_mean;
        fa.noise_idx = noise_idx ? h->c_noise : nullptr;
        fa.noise = hyp_noise(h);
        fa.n_noise = h->n_noise;
        fa.include_noise = include_noise;
        fa.min_var = min_var;
        fa.mean_out = h->c_mu;
        fa.var_out = h->c_var;
        const int nblk = (int)((mc + 255) / 256);
        if (acq) {
            fa.cost_idx = acq->cost_idx ? h->c_cost : nullptr;
            fa.cost = h->acq_par;
            fa.best_f = h->acq_par + acq->n_cost;
            fa.kind_by_cost = h->acq_kind;
            fa.n_cost = acq->n_cost;
            fa.maximize = acq->maximize;
            fa.si = acq->si;
            fa.y_min = acq->y_min;
            fa.y_std = acq->y_std;
            fa.score_out = acq->scores ? h->c_score : nullptr;
            fa.blk_best = h->c_blk_best;
            fa.blk_idx = h->c_blk_idx;
        }
        predict_finish_kernel<<<nblk, 256, 0, h->st>>>(fa);
        CK(cudaGetLastError());
    count_launch();
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
    return predict_impl(h, m, xq, level_idx, noise_idx, mean_idx, include_noise, min_var, mean, var, nullptr);
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
    int rc = predict_impl(h, m, xq, level_idx, nullptr, mean_idx, 0, min_var, nullptr, nullptr, &a);
    if (rc != GPP_OK) return rc;
    if (best_score) *best_score = a.best_score;
    if (best_index) *best_index = a.best_index;
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
