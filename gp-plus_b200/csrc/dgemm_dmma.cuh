// FP64 tensor-core (DMMA m8n8k4) tile GEMM for sm_100a.
//
// One kernel family serves every O(N^3) step of the exact-GP hot path:
//   Cholesky TRSM / SYRK trailing updates, the recursive-doubling triangular inverse and
//   K^-1 = L^-T L^-1 (replacing torch.linalg.cholesky + autograd's cholesky_backward that the
//   reference reaches through gpytorch, optim/mll_scipy.py:37-39,123).
//
//   C[ti,tj] = beta*C[ti,tj] + alpha * sum_{kb in [klo,khi)} A(ti,kb) * B(tj,kb)^T
//
// with 128x128 output tiles, operands in either "k-contiguous" ([row][k]) or
// "k-strided" ([k][row]) row-major layout, a per-tile K range that can depend on the tile
// row / column (triangular operands are skipped, not multiplied by zeros), an optional
// lower-triangle tile filter and a batch dimension.  tcgen05 has no FP64 kind, so the
// tensor-core path for doubles on Blackwell is mma.sync DMMA; sm_100a lowers every f64
// mma shape to DMMA.8x8x4 (checked with cuobjdump), which is what is issued here.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>

namespace gpp {

// process-wide count of kernel launches issued by this library (reported by gpp_launch_count)
inline std::atomic<long long> g_launches{0};
inline thread_local long long t_launches = 0;  // same count per host thread (graph-capture accounting)
inline void count_launch(int k = 1) {
    g_launches.fetch_add(k, std::memory_order_relaxed);
    t_launches += k;
}

constexpr int TILE = 128;        // output tile edge and K block
constexpr int BK = 16;           // k-chunk staged per pipeline stage
constexpr int LDS_KC = BK + 4;   // [row][k] smem row stride (doubles): banks (8g+2t) conflict-free

// Two CTA shapes share one kernel body.  BM = 128: one 128x128 output tile per CTA (256 threads,
// 4 stages, 160 KB, one CTA per SM).  BM = 64: half a tile (64 rows x 128 cols, 128 threads, 3 stages,
// 90 KB) so that two CTAs are resident per SM and one computes while the other sits at a barrier or
// in its epilogue.
template <int BM>
struct GemmCfg {
    static constexpr int THREADS = BM * 2;
    static constexpr int STAGES = (BM == 128) ? 4 : 3;
    static constexpr int A_LDS_KS = BM + 4;     // [k][row] smem row stride of the A operand
    static constexpr int B_LDS_KS = TILE + 4;   // [k][row] smem row stride of the B operand
    static constexpr int A_STAGE = (BM * LDS_KC > BK * A_LDS_KS) ? BM * LDS_KC : BK * A_LDS_KS;
    static constexpr int B_STAGE = (TILE * LDS_KC > BK * B_LDS_KS) ? TILE * LDS_KC : BK * B_LDS_KS;
    static constexpr int SMEM_BYTES = STAGES * (A_STAGE + B_STAGE) * 8;
    static constexpr int MIN_CTAS = (BM == 128) ? 1 : 2;
};

constexpr int GEMM_BM = 64;         // CTA shape of launch_gemm
constexpr int GEMM_NUM_SMS = 148;   // B200
constexpr int GEMM_STAGGER = 10;    // phase shift of the two resident CTAs of an SM in tenths of half a tile time:
                                    // potrf alone 53.4 -> 52.4 ms at N = 16384

enum KSel { KSEL_CONST = 0, KSEL_TI = 1, KSEL_TJ = 2 };
enum TileMap { MAP_RECT = 0, MAP_TRI = 1 };
// EPI_STORE_ROWSQ: the EPI_ROWSQ row sums (same values, bit for bit) and the plain EPI_STORE tile (alpha = 1, beta = 0
// assumed by the caller), for prediction gradients that need U = K* L^-T itself
enum Epilogue { EPI_STORE = 0, EPI_ROWSQ = 2, EPI_STORE_ROWSQ = 3 };

struct GemmOp {
    const double* A;
    const double* B;
    double* C;
    int lda, ldb, ldc;
    long long a_zs, b_zs, c_zs;  // batch strides in elements
    int tiles_m, tiles_n;        // region size in tiles
    int tiles_m_last;            // tiles_m of the last batch entry
    int map;                     // TileMap
    int lower_filter;            // rect map: keep tile iff ti + lower_off >= tj
    int lower_off;
    int klo_sel, klo_c;          // K range in 128-blocks: klo = klo_c + sel(ti|tj)
    int khi_sel, khi_c;          //                         khi = khi_c + sel(ti|tj)
    double alpha, beta;
    int mirror;                  // also store the transposed tile at (tj,ti) (K^-1 full storage)
    int epilogue;                // Epilogue
    double* rowsq;               // EPI_ROWSQ: rowsq[tj * rowsq_ld + global_row] = sum_n acc[row][n]^2
    int rowsq_ld;
    int total_ctas;              // set by launch_gemm: work items along x; CTAs stride over them (persistent when
                                 // the grid is smaller than this)
    int max_ctas;                // 0 = one CTA per work item; otherwise cap on gridDim.x (leaves SMs to other streams)
    int stagger_ns;              // > 0: the second resident CTA of every SM starts this many ns late (see launch_gemm)
};

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
    unsigned s = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
    asm volatile("cp.async.wait_group %0;\n" ::"n"(N));
}

__device__ __forceinline__ void dmma884(double& c0, double& c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
                 : "+d"(c0), "+d"(c1)
                 : "d"(a), "d"(b));
}

// stage one R x BK operand chunk into shared memory with 16-byte cp.async (TH threads)
template <bool KC, int R, int TH>
__device__ __forceinline__ void load_chunk(double* sm, const double* g, int ld, int tid) {
    constexpr int PIECES = R * 8 / TH;  // 16-byte pieces per thread
    if (KC) {
        // global: row r (R rows), 16 contiguous doubles -> 8 x 16B per row
#pragma unroll
        for (int i = 0; i < PIECES; i++) {
            int c = tid + i * TH;
            int r = c >> 3, q = c & 7;
            cp_async16(sm + r * LDS_KC + q * 2, g + (long long)r * ld + q * 2);
        }
    } else {
        // global: k row (16 rows), R contiguous doubles -> R/2 x 16B per row
        constexpr int PPR = R / 2;
#pragma unroll
        for (int i = 0; i < PIECES; i++) {
            int c = tid + i * TH;
            int r = c / PPR, q = c - r * PPR;
            cp_async16(sm + r * (R + 4) + q * 2, g + (long long)r * ld + q * 2);
        }
    }
}

template <bool A_KC, bool B_KC, int BM>
__global__ void __launch_bounds__(GemmCfg<BM>::THREADS, GemmCfg<BM>::MIN_CTAS) dgemm_dmma_kernel(const GemmOp op) {
    using Cfg = GemmCfg<BM>;
    constexpr int NTH = Cfg::THREADS;
    constexpr int NST = Cfg::STAGES;
    constexpr int SPLIT = TILE / BM;  // CTAs per 128-row tile
    extern __shared__ __align__(16) double smem[];
    const int tid = threadIdx.x;
    const int z = blockIdx.y;
    const int tm = (z == (int)gridDim.y - 1) ? op.tiles_m_last : op.tiles_m;
    if (op.stagger_ns > 0 && blockIdx.x >= GEMM_NUM_SMS && blockIdx.x < 2 * GEMM_NUM_SMS) {
        // Two CTAs share an SM so that one computes while the other is in its prologue / epilogue -- which only works
        // if they are out of phase.  With a uniform K range every tile takes the same time, the two CTAs that start
        // together on an SM stay in lock step for the whole launch and reach their epilogues simultaneously.  Delaying
        // the CTAs that fill the second slot of every SM by half a tile time once puts the pair (and every CTA that
        // later inherits one of the two slots) out of phase.
        for (int w = op.stagger_ns; w > 0; w -= 1000) __nanosleep(w > 1000 ? 1000 : w);
    }
  for (int work = blockIdx.x; work < op.total_ctas; work += gridDim.x) {
    const int half = (SPLIT == 1) ? 0 : (work % SPLIT);
    const int tile_id = (SPLIT == 1) ? work : (work / SPLIT);
    const int r0 = half * BM;  // first row of this CTA inside its 128-row tile

    // Tile rasterisation: super-rows of GS tile rows, column-major inside a super-row, so that the ~150 tiles in
    // flight share GS row panels and ~150/GS column panels instead of one row panel and ~150 column panels
    // (LAUUM at N=16384 read 21 GB from DRAM for 3.2 GB of algorithmic traffic with the plain row-major order).
    constexpr int GS = 8;
    int ti, tj;
    if (op.map == MAP_TRI) {
        // lower tiles (tj <= ti); super-row gq holds rows [GS*gq, GS*gq + R), tiles before it: r0g (r0g + 1) / 2
        const int bid = tile_id;
        int gq = (int)((sqrt(8.0 * (double)bid + 1.0) - 1.0) * 0.5) / GS;
        while ((long long)(gq + 1) * GS * ((gq + 1) * GS + 1) / 2 <= bid) gq++;
        while ((long long)gq * GS * (gq * GS + 1) / 2 > bid) gq--;
        const int r0g = gq * GS;
        const int R = (op.tiles_m - r0g < GS) ? (op.tiles_m - r0g) : GS;
        int local = bid - (int)((long long)r0g * (r0g + 1) / 2);
        const int rect = r0g * R;  // full columns 0 .. r0g-1, R tiles each
        if (local < rect) {
            tj = local / R;
            ti = r0g + (local - tj * R);
        } else {
            local -= rect;
            int c = 0;  // triangular corner: column r0g + c holds rows r0g + c .. r0g + R - 1
            while (local >= R - c) { local -= R - c; c++; }
            tj = r0g + c;
            ti = r0g + c + local;
        }
        if (ti >= tm) continue;
    } else {
        const int r0g = (tile_id / (GS * op.tiles_n)) * GS;
        const int R = (op.tiles_m - r0g < GS) ? (op.tiles_m - r0g) : GS;
        const int local = tile_id - r0g * op.tiles_n;
        tj = local / R;
        ti = r0g + (local - tj * R);
        if (ti >= tm) continue;
        if (op.lower_filter && (ti + op.lower_off < tj)) continue;
    }

    int klo = op.klo_c + (op.klo_sel == KSEL_TI ? ti : (op.klo_sel == KSEL_TJ ? tj : 0));
    int khi = op.khi_c + (op.khi_sel == KSEL_TI ? ti : (op.khi_sel == KSEL_TJ ? tj : 0));
    const int nch = (khi > klo) ? (khi - klo) * (TILE / BK) : 0;

    const double* Ag = op.A + (long long)z * op.a_zs;
    const double* Bg = op.B + (long long)z * op.b_zs;
    long long a_step, b_step;  // pointer advance per k-chunk
    if (A_KC) { Ag += ((long long)ti * TILE + r0) * op.lda + (long long)klo * TILE; a_step = BK; }
    else      { Ag += (long long)klo * TILE * op.lda + (long long)ti * TILE + r0; a_step = (long long)BK * op.lda; }
    if (B_KC) { Bg += (long long)tj * TILE * op.ldb + (long long)klo * TILE; b_step = BK; }
    else      { Bg += (long long)klo * TILE * op.ldb + (long long)tj * TILE; b_step = (long long)BK * op.ldb; }

    double* sA = smem;
    double* sB = smem + NST * Cfg::A_STAGE;

    const int warp = tid >> 5, lane = tid & 31;
    const int g = lane >> 2, t = lane & 3;
    const int wm0 = (warp >> 1) * 32;  // BM/32 warps along M
    const int wn0 = (warp & 1) * 64;   // 2 warps along N

    double acc[4][8][2];
#pragma unroll
    for (int i = 0; i < 4; i++)
#pragma unroll
        for (int j = 0; j < 8; j++) { acc[i][j][0] = 0.0; acc[i][j][1] = 0.0; }

    // prologue: S-1 chunks in flight
#pragma unroll
    for (int s = 0; s < NST - 1; s++) {
        if (s < nch) {
            load_chunk<A_KC, BM, NTH>(sA + s * Cfg::A_STAGE, Ag + s * a_step, op.lda, tid);
            load_chunk<B_KC, TILE, NTH>(sB + s * Cfg::B_STAGE, Bg + s * b_step, op.ldb, tid);
        }
        cp_async_commit();
    }

    for (int c = 0; c < nch; c++) {
        cp_async_wait<NST - 2>();
        __syncthreads();
        {
            int cn = c + NST - 1;
            if (cn < nch) {
                int s = cn % NST;
                load_chunk<A_KC, BM, NTH>(sA + s * Cfg::A_STAGE, Ag + cn * a_step, op.lda, tid);
                load_chunk<B_KC, TILE, NTH>(sB + s * Cfg::B_STAGE, Bg + cn * b_step, op.ldb, tid);
            }
            cp_async_commit();
        }
        const double* a_s = sA + (c % NST) * Cfg::A_STAGE;
        const double* b_s = sB + (c % NST) * Cfg::B_STAGE;
#pragma unroll
        for (int kk = 0; kk < BK / 4; kk++) {
            double af[4], bf[8];
#pragma unroll
            for (int mi = 0; mi < 4; mi++) {
                if (A_KC) af[mi] = a_s[(wm0 + mi * 8 + g) * LDS_KC + kk * 4 + t];
                else      af[mi] = a_s[(kk * 4 + t) * Cfg::A_LDS_KS + wm0 + mi * 8 + g];
            }
#pragma unroll
            for (int ni = 0; ni < 8; ni++) {
                if (B_KC) bf[ni] = b_s[(wn0 + ni * 8 + g) * LDS_KC + kk * 4 + t];
                else      bf[ni] = b_s[(kk * 4 + t) * Cfg::B_LDS_KS + wn0 + ni * 8 + g];
            }
#pragma unroll
            for (int mi = 0; mi < 4; mi++)
#pragma unroll
                for (int ni = 0; ni < 8; ni++) dmma884(acc[mi][ni][0], acc[mi][ni][1], af[mi], bf[ni]);
        }
    }
    cp_async_wait<0>();
    __syncthreads();  // every operand read of this CTA is complete (C may alias A)

    const double alpha = op.alpha, beta = op.beta;
    constexpr bool STORE_ROWSQ = A_KC && B_KC;  // EPI_STORE_ROWSQ exists in the K* L^-T instantiation only
    if (op.epilogue == EPI_ROWSQ || (STORE_ROWSQ && op.epilogue == EPI_STORE_ROWSQ)) {
        // rowsq[tj][row] = sum over the tile's 128 columns of (alpha*acc)^2 ; reduce t-lanes then the 2 N-warps
        double* red = smem;  // [2][BM]
#pragma unroll
        for (int mi = 0; mi < 4; mi++) {
            double s = 0.0;
#pragma unroll
            for (int ni = 0; ni < 8; ni++) {
                double v0 = alpha * acc[mi][ni][0], v1 = alpha * acc[mi][ni][1];
                s = fma(v0, v0, s);
                s = fma(v1, v1, s);
            }
            s += __shfl_xor_sync(0xffffffffu, s, 1);
            s += __shfl_xor_sync(0xffffffffu, s, 2);
            if (t == 0) red[(warp & 1) * BM + wm0 + mi * 8 + g] = s;
        }
        __syncthreads();
        if (tid < BM) {
            double s = red[tid] + red[BM + tid];
            op.rowsq[(long long)tj * op.rowsq_ld + (long long)z * op.c_zs + (long long)ti * TILE + r0 + tid] = s;
        }
        __syncthreads();  // `red` aliases the first pipeline stage of the next work item
        if (!STORE_ROWSQ || op.epilogue == EPI_ROWSQ) continue;
    }

    double* Cg = op.C + (long long)z * op.c_zs + ((long long)ti * TILE + r0) * op.ldc + (long long)tj * TILE;
    double* Ct = op.C + (long long)z * op.c_zs + (long long)tj * TILE * op.ldc + (long long)ti * TILE + r0;
    const bool do_mirror = op.mirror && (ti != tj);
#pragma unroll
    for (int mi = 0; mi < 4; mi++) {
#pragma unroll
        for (int ni = 0; ni < 8; ni++) {
            int r = wm0 + mi * 8 + g;
            int cidx = wn0 + ni * 8 + 2 * t;
            double2* p = reinterpret_cast<double2*>(Cg + (long long)r * op.ldc + cidx);
            double2 v;
            v.x = alpha * acc[mi][ni][0];
            v.y = alpha * acc[mi][ni][1];
            if (beta != 0.0) {
                double2 o = *p;
                v.x = fma(beta, o.x, v.x);
                v.y = fma(beta, o.y, v.y);
            }
            *p = v;
            if (do_mirror) {
                Ct[(long long)cidx * op.ldc + r] = v.x;
                Ct[(long long)(cidx + 1) * op.ldc + r] = v.y;
            }
        }
    }
  }  // work items
}

template <int BM>
inline cudaError_t launch_gemm_bm(const GemmOp& op_in, bool a_kc, bool b_kc, int nt, int nbatch, cudaStream_t st) {
    using Cfg = GemmCfg<BM>;
    GemmOp op = op_in;
    op.total_ctas = nt * (TILE / BM);
    int gx = op.total_ctas;
    if (op.max_ctas > 0 && gx > op.max_ctas) gx = op.max_ctas;
    dim3 grid(gx, nbatch), block(Cfg::THREADS);
    if (a_kc && b_kc) dgemm_dmma_kernel<true, true, BM><<<grid, block, Cfg::SMEM_BYTES, st>>>(op);
    else if (a_kc && !b_kc) dgemm_dmma_kernel<true, false, BM><<<grid, block, Cfg::SMEM_BYTES, st>>>(op);
    else if (!a_kc && !b_kc) dgemm_dmma_kernel<false, false, BM><<<grid, block, Cfg::SMEM_BYTES, st>>>(op);
    else dgemm_dmma_kernel<false, true, BM><<<grid, block, Cfg::SMEM_BYTES, st>>>(op);
    return cudaGetLastError();
}

inline cudaError_t launch_gemm(const GemmOp& op, bool a_kc, bool b_kc, int nbatch, cudaStream_t st) {
    int nt;
    if (op.map == MAP_TRI) nt = op.tiles_m * (op.tiles_m + 1) / 2;
    else nt = op.tiles_m * op.tiles_n;
    if (nt <= 0 || nbatch <= 0) return cudaSuccess;
    count_launch();
    if (nbatch == 1 && op.klo_sel == KSEL_CONST && op.khi_sel == KSEL_CONST && 2 * nt >= 16 * GEMM_NUM_SMS &&
        op.max_ctas == 0) {
        // uniform K, at least eight waves: half a tile time = (khi - klo) * 8 chunks * ~2.2 us per chunk / 2
        GemmOp o2 = op;
        o2.stagger_ns = (op.khi_c - op.klo_c) * 8 * 11 * GEMM_STAGGER * 10;
        return launch_gemm_bm<GEMM_BM>(o2, a_kc, b_kc, nt, nbatch, st);
    }
    return launch_gemm_bm<GEMM_BM>(op, a_kc, b_kc, nt, nbatch, st);
}

template <int BM>
inline cudaError_t gemm_set_attributes_bm() {
    cudaError_t e;
    const int b = GemmCfg<BM>::SMEM_BYTES;
    e = cudaFuncSetAttribute(dgemm_dmma_kernel<true, true, BM>, cudaFuncAttributeMaxDynamicSharedMemorySize, b);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(dgemm_dmma_kernel<true, false, BM>, cudaFuncAttributeMaxDynamicSharedMemorySize, b);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(dgemm_dmma_kernel<false, false, BM>, cudaFuncAttributeMaxDynamicSharedMemorySize, b);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(dgemm_dmma_kernel<false, true, BM>, cudaFuncAttributeMaxDynamicSharedMemorySize, b);
    return e;
}

inline cudaError_t gemm_set_attributes() { return gemm_set_attributes_bm<GEMM_BM>(); }

inline GemmOp gemm_default() {
    GemmOp op{};
    op.alpha = 1.0;
    op.beta = 0.0;
    op.map = MAP_RECT;
    op.klo_sel = KSEL_CONST;
    op.khi_sel = KSEL_CONST;
    op.tiles_n = 1;
    op.epilogue = EPI_STORE;
    return op;
}

}  // namespace gpp
