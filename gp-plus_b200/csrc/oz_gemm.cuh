// FP64-equivalent tile GEMM on the INT8 tcgen05 tensor cores ("Ozaki" splitting), sm_100a.
//
// tcgen05 has no FP64 kind, and the exact DMMA path (dgemm_dmma.cuh) tops out at ~35 TFLOP/s.  The three O(N^3)
// stages of the evaluation (trailing updates of the factorisation, the levels of the triangular inverse and
// K^-1 = L^-T L^-1; reference: torch.linalg.cholesky + cholesky_backward reached through
// MultivariateNormal.log_prob, optim/mll_scipy.py:37-39,123) can instead run as exact integer GEMMs:
//
//   every operand row r is scaled by a power of two, x = 2^e_r * sum_{p<7} d_p 256^-(p+1) (+ < 2^(e_r-56)),
//   d_p signed base-256 digits ("digit planes", int8, written by oz_split.cuh), and
//
//   C[r,c] = beta C[r,c] + alpha 2^(ea_r + eb_c) sum_{lvl<7} 256^-(lvl+2) sum_{i+j=lvl} sum_k A_i[r,k] B_j[c,k]
//
//   (28 plane pairs; the dropped pairs i+j >= 7 are below 2^-54 of |row||col|).  Every level accumulates exactly in
//   its own int32 TMEM accumulator: |d| <= 128, so K <= 16384 per accumulation cannot overflow.
//
// Measured issue rates of tcgen05.mma.kind::i8 at M = 128 (tools/oz_lab rate): N = 64: 48 cycles (shared-memory
// operand reads, 6 KB per MMA at 128 B/clk), N = 128: 64 cycles, N = 256: 128 cycles (both = 4.5 POPS).  N = 128 is
// the narrowest shape that reaches the peak, and TMEM holds four 128-column accumulators, so a 128x128 output tile
// is produced in two passes over K:
//   pass 0: levels 0..2 ( 6 plane pairs, planes 0..2 of both operands),  C  = beta C + alpha * (...)
//   pass 1: levels 3..6 (22 plane pairs, planes 0..6),                   C += alpha * (...)
// (20 plane tiles streamed per K chunk; the 4 + 3 split streams 22 and measured 1-5 % slower in isolation: the kernel
// is bound by the bytes an SM ingests from L2)
//
// One CTA per SM (all of TMEM, 225 KB of shared memory), each looping over a few output tiles:
//   warp 0 (one lane)  TMA producer: per 64-byte K chunk the planes the pass needs (128 rows x 64 B, SWIZZLE_64B),
//                      2-slot mbarrier ring
//   warp 1 (one lane)  tcgen05.mma.cta_group::1.kind::i8, M = N = 128, K = 32 (12 / 44 per slot); tcgen05.commit frees the slot /
//                      publishes the accumulators
//   warps 2-9          epilogue: tcgen05.ld 16x256b (two warps per TMEM lane quarter, 64 columns each; a quad of threads
//                      owns 64 contiguous bytes of a C row), Horner over the levels in FP64, power-of-two row /
//                      column scales, read-modify-write of C in full 32-byte sectors
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "dgemm_dmma.cuh"
#include "tma.cuh"

namespace gpp {

constexpr int OZ_S = 7;            // digit planes per operand
#ifndef GPP_OZ_L0
#define GPP_OZ_L0 3
#endif
constexpr int OZ_L0 = GPP_OZ_L0;   // pass 0: levels 0 .. L0-1 (planes 0 .. L0-1), pass 1: levels L0 .. 6 (all planes)
constexpr int OZ_NACC = (OZ_L0 > OZ_S - OZ_L0) ? OZ_L0 : OZ_S - OZ_L0;   // accumulators live at a time
constexpr int OZ_BM = 128;         // output rows per work item (UMMA M)
constexpr int OZ_BN = 128;         // output columns per work item (UMMA N)
constexpr int OZ_BK = 64;          // K bytes (= int8 elements) per ring slot = swizzle width
constexpr int OZ_STAGES = 2;
constexpr int OZ_UMMA_K = 32;      // K of one kind::i8 MMA
constexpr int OZ_A_TILE = OZ_BM * OZ_BK;                       // 8192 B per plane and slot
constexpr int OZ_B_TILE = OZ_BN * OZ_BK;
constexpr int OZ_STAGE_BYTES = OZ_S * (OZ_A_TILE + OZ_B_TILE); // 114688 (pass 1; pass 0 fills 65536 of it)
constexpr int OZ_SMEM_BYTES = OZ_STAGES * OZ_STAGE_BYTES + 1024 /*alignment slack*/ + 128 /*barriers*/;
constexpr int OZ_EPI_WARPS = 8;
constexpr int OZ_THREADS = 32 * (2 + OZ_EPI_WARPS);
constexpr int OZ_TMEM_COLS = 512;
static_assert(OZ_SMEM_BYTES <= 232448, "oz_gemm shared memory exceeds the 227 KB per-CTA limit");
static_assert(OZ_BK == 32 || OZ_BK == 64 || OZ_BK == 128, "K chunk must equal a swizzle width");
static_assert(OZ_NACC * OZ_BN <= OZ_TMEM_COLS && OZ_L0 >= 1 && OZ_L0 < OZ_S, "accumulators must fit in TMEM");

// same K-range / tile-map vocabulary as GemmOp (dgemm_dmma.cuh); a work item is one 128x128 tile
struct OzGemmOp {
    // digit planes: plane p of A is rows [p * a_plane_rows, (p+1) * a_plane_rows) of tensor map A (inner dim = k)
    int a_plane_rows, b_plane_rows;
    int a_row0, b_row0;              // plane row of tile row / tile column 0
    int a_k0, b_k0;                  // plane k coordinate of K block 0
    int a_zs_row, a_zs_k, b_zs_row, b_zs_k;   // batch steps in plane coordinates
    const double* a_scale;           // 2^ea per plane row (same row coordinate as the planes, batch included)
    const double* b_scale;
    double* C;
    int ldc;
    long long c_zs;
    int tiles_m, tiles_n, tiles_m_last;
    int map, lower_filter, lower_off;
    int klo_sel, klo_c, khi_sel, khi_c;
    int levels;                      // significance levels kept (0 = all 7): pairs with i + j >= levels and the planes they
                                     // alone would need are skipped.  K^-1 feeds only the gradient trace (tolerance 1e-8)
                                     // and runs with 6 (21 pairs); everything that feeds the objective keeps 7
    int k_min, k_max;                // clamp of the K range in 128-blocks (k_max <= 0: none): long accumulations are cut
                                     // into launches of <= 128 blocks so that an int32 accumulator cannot overflow
    double alpha, beta;
    int n_tiles;                     // 128x128 tiles per batch entry (set by launch_oz_gemm)
    int stagger_ns;                  // > 0: CTA b of the first wave starts (b mod 148) / 148 of this many ns late, so that
                                     // CTAs (equal work each) retire evenly spread in time instead of in synchronised
                                     // waves and a higher-priority stream finds a free SM within microseconds
    long long* prof;                 // optional (development): clock64 stamps of CTA 0's first item, 4 per pass:
                                     // accumulators free, MMAs issued, accumulators complete, epilogue done
};

// ---- PTX wrappers -------------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* tm, int c0, int c1, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
            smem_u32(smem_dst)),
        "l"(reinterpret_cast<uint64_t>(tm)), "r"(c0), "r"(c1), "r"(smem_u32(bar))
        : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* tm) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tm)) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst, uint32_t cols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(cols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
// D[tmem] (+)= A[smem] * B[smem]^T, int8 x int8 -> int32
__device__ __forceinline__ void umma_i8(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// arrive on an mbarrier once every tcgen05 operation issued so far by this thread has completed
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}
// 16 consecutive accumulator columns of this thread's TMEM lane
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, int (&v)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr)
        : "memory");
}
// 16 TMEM lanes x 32 columns: register 4j + {0,1} = lane (base + laneid / 4), columns 8j + 2 (laneid % 4) + {0,1};
// register 4j + {2,3} = the same columns of lane (base + 8 + laneid / 4)   (cute SM100_TMEM_LOAD_16dp256b4x layout).
// A quad of threads therefore holds 8 consecutive columns of a row: 64 contiguous bytes once converted to FP64.
__device__ __forceinline__ void tmem_ld_16x256b_x4(uint32_t taddr, int (&v)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.16x256b.x4.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// K-major operand tile, rows of OZ_BK bytes, SWIZZLE_<OZ_BK>B: 8-row groups are 8 * OZ_BK bytes apart (SBO), LBO unused
__device__ __forceinline__ uint64_t oz_smem_desc(uint32_t smem_addr) {
    constexpr uint64_t layout = (OZ_BK == 128) ? 2 : (OZ_BK == 64 ? 4 : 6);
    return (uint64_t)((smem_addr & 0x3FFFF) >> 4) | ((uint64_t)((8 * OZ_BK) >> 4) << 32) | (1ull << 46) | (layout << 61);
}
// kind::i8 instruction descriptor: D = s32, A = B = signed 8 bit, both K-major, M = 128, N = 64
constexpr uint32_t OZ_IDESC = (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(OZ_BN >> 3) << 17) | ((uint32_t)(OZ_BM >> 4) << 24);

// work item -> (ti, tj); false: filtered out.  Lower-triangular map in super-rows of GS tile rows like the DMMA
// kernel, so that the items in flight share a few row panels and a few column panels in L2.
__device__ __forceinline__ bool oz_decode(const OzGemmOp& op, int tile_id, int tm, int& ti, int& tj) {
    constexpr int GS = 8;
    if (op.map == MAP_TRI) {
        const int bid = tile_id;
        int gq = (int)((sqrt(8.0 * (double)bid + 1.0) - 1.0) * 0.5) / GS;
        while ((long long)(gq + 1) * GS * ((gq + 1) * GS + 1) / 2 <= bid) gq++;
        while ((long long)gq * GS * (gq * GS + 1) / 2 > bid) gq--;
        const int r0g = gq * GS;
        const int R = (op.tiles_m - r0g < GS) ? (op.tiles_m - r0g) : GS;
        int local = bid - (int)((long long)r0g * (r0g + 1) / 2);
        const int rect = r0g * R;
        if (local < rect) {
            tj = local / R;
            ti = r0g + (local - tj * R);
        } else {
            local -= rect;
            int c = 0;
            while (local >= R - c) { local -= R - c; c++; }
            tj = r0g + c;
            ti = r0g + c + local;
        }
        return ti < tm;
    }
    const int r0g = (tile_id / (GS * op.tiles_n)) * GS;
    const int R = (op.tiles_m - r0g < GS) ? (op.tiles_m - r0g) : GS;
    const int local = tile_id - r0g * op.tiles_n;
    tj = local / R;
    ti = r0g + (local - tj * R);
    if (ti >= tm) return false;
    if (op.lower_filter && (ti + op.lower_off < tj)) return false;
    return true;
}
__device__ __forceinline__ int oz_chunks(const OzGemmOp& op, int ti, int tj, int& klo) {
    klo = op.klo_c + (op.klo_sel == KSEL_TI ? ti : (op.klo_sel == KSEL_TJ ? tj : 0));
    int khi = op.khi_c + (op.khi_sel == KSEL_TI ? ti : (op.khi_sel == KSEL_TJ ? tj : 0));
    if (op.k_max > 0) {
        klo = klo > op.k_min ? klo : op.k_min;
        khi = khi < op.k_max ? khi : op.k_max;
    }
    return (khi > klo) ? (khi - klo) * (TILE / OZ_BK) : 0;
}

__global__ void __launch_bounds__(OZ_THREADS, 1)
oz_gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const OzGemmOp op) {
    extern __shared__ uint8_t oz_smem_raw[];
    uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(oz_smem_raw) + 1023) & ~(uintptr_t)1023);
    uint64_t* bars = reinterpret_cast<uint64_t*>(base + OZ_STAGES * OZ_STAGE_BYTES);
    uint64_t* full = bars;                          // [OZ_STAGES] TMA -> MMA
    uint64_t* empty = bars + OZ_STAGES;             // [OZ_STAGES] MMA -> TMA
    uint64_t* tmem_full = bars + 2 * OZ_STAGES;     // MMA -> epilogue
    uint64_t* tmem_empty = bars + 2 * OZ_STAGES + 1;  // epilogue -> MMA
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * OZ_STAGES + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int z = blockIdx.y;
    const int tm = (z == (int)gridDim.y - 1) ? op.tiles_m_last : op.tiles_m;
    const int n_items = op.n_tiles;
    const int nlev = (op.levels > OZ_L0 && op.levels < OZ_S) ? op.levels : OZ_S;   // levels kept (pass 1: planes 0 .. nlev-1)
    if (op.stagger_ns > 0 && blockIdx.x < GEMM_NUM_SMS) {
        for (int w = (int)((long long)blockIdx.x * op.stagger_ns / GEMM_NUM_SMS); w > 0; w -= 1000)
            __nanosleep(w > 1000 ? 1000 : w);
    }

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&tmA);
        tma_prefetch_desc(&tmB);
        for (int s = 0; s < OZ_STAGES; s++) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], 1);
        }
        mbar_init(tmem_full, 1);
        mbar_init(tmem_empty, OZ_EPI_WARPS);
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc(tmem_slot, OZ_TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ===== TMA producer =====
        if (lane == 0) {
            uint32_t stage = 0, phase = 0;
            for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
                int ti, tj, klo;
                if (!oz_decode(op, item, tm, ti, tj)) continue;
                const int nch = oz_chunks(op, ti, tj, klo);
                const int a_row = op.a_row0 + z * op.a_zs_row + ti * TILE;
                const int b_row = op.b_row0 + z * op.b_zs_row + tj * TILE;
                const int ka = op.a_k0 + z * op.a_zs_k + klo * TILE;
                const int kb = op.b_k0 + z * op.b_zs_k + klo * TILE;
                for (int pass = 0; pass < 2; pass++) {
                    const int npl = pass == 0 ? OZ_L0 : nlev;
                    for (int c = 0; c < nch; c++) {
                        mbar_wait(&empty[stage], phase ^ 1);
                        mbar_arrive_expect_tx(&full[stage], (uint32_t)npl * (OZ_A_TILE + OZ_B_TILE));
                        uint8_t* sa = base + stage * OZ_STAGE_BYTES;
                        uint8_t* sb = sa + OZ_S * OZ_A_TILE;
                        for (int p = 0; p < npl; p++) {
                            tma_load_2d(sa + p * OZ_A_TILE, &tmA, ka + c * OZ_BK, p * op.a_plane_rows + a_row, &full[stage]);
                            tma_load_2d(sb + p * OZ_B_TILE, &tmB, kb + c * OZ_BK, p * op.b_plane_rows + b_row, &full[stage]);
                        }
                        if (++stage == OZ_STAGES) { stage = 0; phase ^= 1; }
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer =====
        uint32_t stage = 0, phase = 0, tphase = 0;
        for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
            int ti, tj, klo;
            if (!oz_decode(op, item, tm, ti, tj)) continue;
            const int nch = oz_chunks(op, ti, tj, klo);
            if (nch == 0) continue;
            for (int pass = 0; pass < 2; pass++) {
                mbar_wait(tmem_empty, tphase ^ 1);   // the epilogue has drained the previous accumulators
                tc_fence_after();
                if (op.prof && blockIdx.x == 0 && z == 0 && item == 0 && lane == 0) op.prof[pass * 4 + 0] = clock64();
                for (int c = 0; c < nch; c++) {
                    mbar_wait(&full[stage], phase);
                    tc_fence_after();
                    if (lane == 0) {
                        const uint32_t sa = smem_u32(base + stage * OZ_STAGE_BYTES);
                        const uint32_t sb = sa + OZ_S * OZ_A_TILE;
                        if (pass == 0) {
#pragma unroll
                            for (int ks = 0; ks < OZ_BK / OZ_UMMA_K; ks++) {
#pragma unroll
                                for (int lvl = 0; lvl < OZ_L0; lvl++) {
#pragma unroll
                                    for (int i = 0; i <= lvl; i++) {
                                        const int j = lvl - i;
                                        const uint64_t ad = oz_smem_desc(sa + i * OZ_A_TILE + ks * OZ_UMMA_K);
                                        const uint64_t bd = oz_smem_desc(sb + j * OZ_B_TILE + ks * OZ_UMMA_K);
                                        umma_i8(tmem_base + lvl * OZ_BN, ad, bd, OZ_IDESC, (c > 0 || ks > 0 || i > 0) ? 1u : 0u);
                                    }
                                }
                            }
                        } else {
#pragma unroll
                            for (int ks = 0; ks < OZ_BK / OZ_UMMA_K; ks++) {
#pragma unroll
                                for (int lvl = OZ_L0; lvl < OZ_S; lvl++) {
#pragma unroll
                                    for (int i = 0; i <= lvl; i++) {
                                        const int j = lvl - i;
                                        if (i < OZ_S && j < OZ_S && lvl < nlev) {
                                            const uint64_t ad = oz_smem_desc(sa + i * OZ_A_TILE + ks * OZ_UMMA_K);
                                            const uint64_t bd = oz_smem_desc(sb + j * OZ_B_TILE + ks * OZ_UMMA_K);
                                            umma_i8(tmem_base + (lvl - OZ_L0) * OZ_BN, ad, bd, OZ_IDESC,
                                                    (c > 0 || ks > 0 || i > 0) ? 1u : 0u);
                                        }
                                    }
                                }
                            }
                        }
                        umma_commit(&empty[stage]);                 // slot reusable once these MMAs have read it
                        if (c == nch - 1) umma_commit(tmem_full);   // accumulators of this pass complete
                    }
                    __syncwarp();
                    if (++stage == OZ_STAGES) { stage = 0; phase ^= 1; }
                }
                if (op.prof && blockIdx.x == 0 && z == 0 && item == 0 && lane == 0) op.prof[pass * 4 + 1] = clock64();
                tphase ^= 1;
            }
        }
    } else {
        // ===== epilogue: TMEM lane quarter (warp % 4), 64 columns per warp; 16-lane x 32-column loads whose fragment
        // layout gives every quad of threads 64 contiguous bytes of a C row (full 32-byte sectors both ways) =====
        const int q = warp & 3;
        const int ch = (warp - 2) >> 2;
        const int r_in = lane >> 2, cq = (lane & 3) * 2;
        uint32_t tphase = 0;
        for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
            int ti, tj, klo;
            if (!oz_decode(op, item, tm, ti, tj)) continue;
            const int nch = oz_chunks(op, ti, tj, klo);
            // this thread's first element of the tile: row q*32 + r_in, column ch*64 + cq
            double* C0 = op.C + (long long)z * op.c_zs + ((long long)ti * TILE + q * 32 + r_in) * op.ldc + (long long)tj * TILE +
                         ch * 64 + cq;
            const double alpha = op.alpha;
            if (nch == 0) {
                // empty K range: C <- beta C
                const double beta = op.beta;
                for (int rr = 0; rr < 4; rr++)
                    for (int j = 0; j < 8; j++) {
                        double2* p2 = reinterpret_cast<double2*>(C0 + (long long)rr * 8 * op.ldc + 8 * j);
                        double2 o = make_double2(0.0, 0.0);
                        if (beta != 0.0) { o = *p2; o.x *= beta; o.y *= beta; }
                        *p2 = o;
                    }
                continue;
            }
            const double* sap = op.a_scale + op.a_row0 + z * op.a_zs_row + ti * TILE + q * 32 + r_in;
            const double* sbp = op.b_scale + op.b_row0 + z * op.b_zs_row + tj * TILE + ch * 64 + cq;
            for (int pass = 0; pass < 2; pass++) {
                const double beta = pass == 0 ? op.beta : 1.0;
                // 256^-(lvl+2) of the pass's lowest level: 2^-16 (pass 0), 2^-(16 + 8 L0) (pass 1)
                const double ps = alpha * (pass == 0 ? (1.0 / 65536.0) : (1.0 / 65536.0) / (double)(1ull << (8 * OZ_L0)));
                // step = (row half rh, 32-column group cg): rows q*32 + 16 rh + r_in + {0, 8}, columns 32 cg + 8 j + cq + {0,1}.
                // C and the scales of a step are fetched one step ahead (for the first step: before the pass's MMAs
                // have finished), so that their latency is not paid per element
                double2 old[8], sb2[4];
                double sA, sB;
                auto prefetch = [&](int step) {
                    const int rh = step >> 1, cg = step & 1;
                    sA = sap[rh * 16] * ps;
                    sB = sap[rh * 16 + 8] * ps;
                    const double* crow = C0 + (long long)(rh * 16) * op.ldc + cg * 32;
#pragma unroll
                    for (int j = 0; j < 4; j++) {
                        sb2[j] = *reinterpret_cast<const double2*>(sbp + cg * 32 + 8 * j);
                        if (beta != 0.0) {
                            old[2 * j] = *reinterpret_cast<const double2*>(crow + 8 * j);
                            old[2 * j + 1] = *reinterpret_cast<const double2*>(crow + (long long)8 * op.ldc + 8 * j);
                        } else {
                            old[2 * j] = make_double2(0.0, 0.0);
                            old[2 * j + 1] = make_double2(0.0, 0.0);
                        }
                    }
                };
                prefetch(0);
                mbar_wait(tmem_full, tphase);
                tc_fence_after();
                if (op.prof && blockIdx.x == 0 && z == 0 && item == 0 && threadIdx.x == 64) op.prof[pass * 4 + 2] = clock64();
#pragma unroll 1
                for (int step = 0; step < 4; step++) {
                    const int rh = step >> 1, cg = step & 1;
                    const uint32_t taddr = tmem_base + ((uint32_t)(q * 32 + rh * 16) << 16) + ch * 64 + cg * 32;
                    int v[OZ_NACC][16];
                    if (pass == 0) {
#pragma unroll
                        for (int a = 0; a < OZ_L0; a++) tmem_ld_16x256b_x4(taddr + a * OZ_BN, v[a]);
#pragma unroll
                        for (int a = OZ_L0; a < OZ_NACC; a++)
#pragma unroll
                            for (int e = 0; e < 16; e++) v[a][e] = 0;
                    } else {
#pragma unroll
                        for (int a = 0; a < OZ_S - OZ_L0; a++) {
                            if (OZ_L0 + a < nlev) {
                                tmem_ld_16x256b_x4(taddr + a * OZ_BN, v[a]);
                            } else {
#pragma unroll
                                for (int e = 0; e < 16; e++) v[a][e] = 0;
                            }
                        }
#pragma unroll
                        for (int a = OZ_S - OZ_L0; a < OZ_NACC; a++)
#pragma unroll
                            for (int e = 0; e < 16; e++) v[a][e] = 0;
                    }
                    tmem_ld_wait();
                    double2 o[8];
#pragma unroll
                    for (int j = 0; j < 4; j++) {
#pragma unroll
                        for (int h = 0; h < 2; h++) {   // h = 0: row r_in, h = 1: row r_in + 8
                            double s0 = (double)v[OZ_NACC - 1][4 * j + 2 * h], s1 = (double)v[OZ_NACC - 1][4 * j + 2 * h + 1];
#pragma unroll
                            for (int a = OZ_NACC - 2; a >= 0; a--) {
                                s0 = fma(s0, 1.0 / 256.0, (double)v[a][4 * j + 2 * h]);
                                s1 = fma(s1, 1.0 / 256.0, (double)v[a][4 * j + 2 * h + 1]);
                            }
                            const double sr = h == 0 ? sA : sB;
                            o[2 * j + h].x = fma(beta, old[2 * j + h].x, s0 * sr * sb2[j].x);
                            o[2 * j + h].y = fma(beta, old[2 * j + h].y, s1 * sr * sb2[j].y);
                        }
                    }
                    double* crow = C0 + (long long)(rh * 16) * op.ldc + cg * 32;
                    if (step + 1 < 4) prefetch(step + 1);
#pragma unroll
                    for (int j = 0; j < 4; j++) {
                        *reinterpret_cast<double2*>(crow + 8 * j) = o[2 * j];
                        *reinterpret_cast<double2*>(crow + (long long)8 * op.ldc + 8 * j) = o[2 * j + 1];
                    }
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(tmem_empty);
                if (op.prof && blockIdx.x == 0 && z == 0 && item == 0 && threadIdx.x == 64) op.prof[pass * 4 + 3] = clock64();
                tphase ^= 1;
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_base, OZ_TMEM_COLS);
}

// ---- host side ----------------------------------------------------------------------------------------------
typedef CUresult (*oz_encode_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                 const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                 CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
inline oz_encode_fn oz_encoder() {
    static oz_encode_fn fn = [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qr;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qr) != cudaSuccess ||
            qr != cudaDriverEntryPointSuccess)
            p = nullptr;
        return reinterpret_cast<oz_encode_fn>(p);
    }();
    return fn;
}

// tensor map over stacked digit planes: inner dimension k (bytes), rows = OZ_S * plane_rows, row pitch `pitch` bytes
inline cudaError_t oz_make_map(CUtensorMap* tm, const int8_t* planes, long long k_extent, long long rows_total,
                               long long pitch, int box_rows) {
    oz_encode_fn enc = oz_encoder();
    if (!enc) return cudaErrorNotSupported;
    cuuint64_t dims[2] = {(cuuint64_t)k_extent, (cuuint64_t)rows_total};
    cuuint64_t strides[1] = {(cuuint64_t)pitch};
    cuuint32_t box[2] = {(cuuint32_t)OZ_BK, (cuuint32_t)box_rows};
    cuuint32_t es[2] = {1, 1};
    const CUtensorMapSwizzle sw = (OZ_BK == 128) ? CU_TENSOR_MAP_SWIZZLE_128B
                                                 : (OZ_BK == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B);
    CUresult r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<int8_t*>(planes), dims, strides, box, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? cudaSuccess : cudaErrorInvalidValue;
}

inline cudaError_t oz_set_attributes() {
    return cudaFuncSetAttribute(oz_gemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, OZ_SMEM_BYTES);
}

// items_per_cta: CTAs are NOT persistent over the whole launch -- each handles about this many 128x128 tiles
// (grid-stride), so that SMs are handed back every few items and higher-priority streams (the panel chain of the
// factorisation) get in; the hardware block scheduler does the load balancing (two per CTA: DESIGN.md section 7).
inline cudaError_t launch_oz_gemm(const CUtensorMap& tmA, const CUtensorMap& tmB, const OzGemmOp& op_in, int nbatch,
                                  cudaStream_t st, int items_per_cta = 1) {
    OzGemmOp op = op_in;
    if (op.map == MAP_TRI) op.n_tiles = op.tiles_m * (op.tiles_m + 1) / 2;
    else op.n_tiles = op.tiles_m * op.tiles_n;
    if (op.n_tiles <= 0 || nbatch <= 0) return cudaSuccess;
    int gx = (op.n_tiles + items_per_cta - 1) / items_per_cta;
    if (gx < 1) gx = 1;
    count_launch();
    oz_gemm_kernel<<<dim3(gx, nbatch), OZ_THREADS, OZ_SMEM_BYTES, st>>>(tmA, tmB, op);
    return cudaGetLastError();
}


// ---- raw tcgen05 kind::i8 issue rate (the roofline denominator of this kernel family) -----------------------------
// One CTA per SM, M = 128 MMAs of width N issued back to back on resident shared-memory tiles (no TMA traffic).
template <int N>
__global__ void __launch_bounds__(128, 1) oz_mma_rate_kernel(int iters) {
    extern __shared__ uint8_t oz_rate_raw[];
    uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(oz_rate_raw) + 1023) & ~(uintptr_t)1023);
    __shared__ uint64_t bar;
    __shared__ uint32_t slot;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    constexpr int TILES = 4;
    for (int i = threadIdx.x; i < TILES * (128 + N) * 64 / 4; i += blockDim.x) reinterpret_cast<uint32_t*>(base)[i] = 0x01ff02feu;
    if (threadIdx.x == 0) {
        mbar_init(&bar, 1);
        fence_barrier_init();
    }
    if (warp == 0) tmem_alloc(&slot, 512);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tm = slot;
    constexpr uint32_t idesc = (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
    if (warp == 1 && lane == 0) {
        const uint32_t sa = smem_u32(base), sb = sa + TILES * 128 * 64;
        constexpr int nacc = 512 / N;
        const uint64_t hi = ((uint64_t)((8 * 64) >> 4) << 32) | (1ull << 46) | (4ull << 61);
        for (int it = 0; it < iters; it += 8) {
#pragma unroll
            for (int u = 0; u < 8; u++) {
                const int ia = (u * 3) % TILES, ib = (u * 5) % TILES;
#pragma unroll
                for (int ks = 0; ks < 2; ks++) {
                    const uint64_t ad = (uint64_t)(((sa + ia * 128 * 64 + ks * 32) & 0x3FFFF) >> 4) | hi;
                    const uint64_t bd = (uint64_t)(((sb + ib * N * 64 + ks * 32) & 0x3FFFF) >> 4) | hi;
                    umma_i8(tm + (u % nacc) * N, ad, bd, idesc, 1u);
                }
            }
        }
        umma_commit(&bar);
        mbar_wait(&bar, 0);
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tm, 512);
}

// int8 tera-ops per second of the whole GPU for MMA width n (64, 128 or 256); 2 * 128 * n * 32 ops per MMA
template <int N>
inline cudaError_t oz_probe_rate_n(int iters, double* tops) {
    constexpr int smem = 4 * (128 + N) * 64 + 2048;
    cudaError_t e = cudaFuncSetAttribute(oz_mma_rate_kernel<N>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e != cudaSuccess) return e;
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    oz_mma_rate_kernel<N><<<GEMM_NUM_SMS, 128, smem>>>(iters);
    double best = 0.0;
    for (int rep = 0; rep < 3; rep++) {
        cudaEventRecord(e0);
        oz_mma_rate_kernel<N><<<GEMM_NUM_SMS, 128, smem>>>(iters);
        cudaEventRecord(e1);
        e = cudaEventSynchronize(e1);
        if (e != cudaSuccess) break;
        float ms = 0.f;
        cudaEventElapsedTime(&ms, e0, e1);
        const double t = (double)GEMM_NUM_SMS * iters * 2.0 * (2.0 * 128.0 * N * 32.0) / (ms * 1e-3) * 1e-12;
        if (t > best) best = t;
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    *tops = best;
    return e;
}

inline OzGemmOp oz_default() {
    OzGemmOp op{};
    op.alpha = 1.0;
    op.beta = 0.0;
    op.map = MAP_RECT;
    op.klo_sel = KSEL_CONST;
    op.khi_sel = KSEL_CONST;
    op.tiles_n = 1;
    return op;
}

}  // namespace gpp
