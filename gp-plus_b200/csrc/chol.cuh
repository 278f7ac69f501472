// Blocked FP64 Cholesky, triangular inverse and K^-1 on top of the DMMA tile GEMM.
//
// Replaces psd_safe_cholesky / torch.linalg.cholesky_ex and the autograd cholesky_backward
// the reference reaches through MultivariateNormal.log_prob (optim/mll_scipy.py:37-39,123;
// SURVEY Appendix A.5).  All matrices are row-major with leading dimension ld = Np, Np a
// multiple of 128 (padded rows/cols carry an identity block, so they change neither the
// factor, log|K| nor the solves).
//
//   1. potrf: right-looking with look-ahead.  A panel (4 or 8 tile columns, factored recursively down to pairs)
//      runs on a high-priority side stream:
//        leaf  (one CTA): L_kk = chol(A_kk) and L_kk^-1 (written into the diagonal block of M)
//        TRSM  (DMMA GEMM, K=128): A_ik <- A_ik * L_kk^-T  via the explicit 128x128 inverse
//        in-panel updates (DMMA GEMM, K = 128 .. panel/2)
//      while the trailing SYRK of the previous panel (DMMA GEMM, K = panel width, lower tiles) runs on the main stream.
//   2. trtri: M = L^-1 by recursive doubling.  With the diagonal 128-blocks already inverted,
//      level h combines aligned groups of h blocks:  M21 = -M22 * (L21 * M11); every group of
//      a level is independent, so a level is two batched GEMM launches (ceil(log2 T) levels).  The part that
//      only needs the leading tile columns of L starts behind the factorisation on a third stream.
//   3. lauum: K^-1 = M^T M, one launch over the lower tiles (the upper triangle is not stored on the hot path).
//
// From N = 3072 the O(N^3) parts of all three steps run as exact integer GEMMs on the INT8 tcgen05 tensor cores
// (oz_gemm.cuh / oz_split.cuh / oz_chol.cuh) when the handle carries an OzCtx: the trailing updates (and, from
// N = 12288, the panel solve of the lazy-panel schedule potrf_lazy, whose diagonal blocks are factored by one
// dataflow launch, block_potrf_kernel), the levels hb >= 4 of the inverse, and K^-1.  Everything latency-bound
// (leaf, TRSM and updates inside a diagonal block, small levels) stays on the DMMA kernels of this file.
#pragma once
#include <stdio.h>
#include <stdlib.h>

#include <vector>

#include "dgemm_dmma.cuh"
#include "oz_chol.cuh"

namespace gpp {

constexpr int LEAF_THREADS = 256;
constexpr int LB = 32;     // sub-block edge inside a 128x128 leaf
constexpr int LLD = 132;   // smem leading dimension: 132 = 4 (mod 16) keeps every DMMA fragment load conflict-free
constexpr int TLD = 36;    // per-warp scratch leading dimension (same residue)
constexpr int PANEL_BLOCKS = 4;   // leaf-level panel: in-panel updates run at K = 128
constexpr int PANEL_BASE = 2;      // widest piece factored with K = 128 in-panel updates (the recursion stops here)
inline int g_panel_blocks = 0;     // look-ahead panel width in 128-columns; 0 = by size (12 from N = 12288, else 4)
constexpr unsigned FULL = 0xffffffffu;

// C(32x32) += A(32x32) * B(32x32) by one warp on DMMA; A(r,k) and B(k,n) are element getters.
// acc[mi][ni][e] holds C(mi*8+g, ni*8+2t+e).
template <class FA, class FB>
__device__ __forceinline__ void warp_mm32(double (&acc)[4][4][2], FA getA, FB getB, int g, int t) {
#pragma unroll
    for (int kk = 0; kk < LB; kk += 4) {
        double af[4], bf[4];
#pragma unroll
        for (int mi = 0; mi < 4; mi++) af[mi] = getA(mi * 8 + g, kk + t);
#pragma unroll
        for (int ni = 0; ni < 4; ni++) bf[ni] = getB(kk + t, ni * 8 + g);
#pragma unroll
        for (int mi = 0; mi < 4; mi++)
#pragma unroll
            for (int ni = 0; ni < 4; ni++) dmma884(acc[mi][ni][0], acc[mi][ni][1], af[mi], bf[ni]);
    }
}

__device__ __forceinline__ void acc_zero(double (&acc)[4][4][2]) {
#pragma unroll
    for (int i = 0; i < 4; i++)
#pragma unroll
        for (int j = 0; j < 4; j++) { acc[i][j][0] = 0.0; acc[i][j][1] = 0.0; }
}

// ---------------------------------------------------------------------------------------------
// Leaf: A_kk -> L_kk in place, M_kk <- L_kk^-1, logdet_part[kb] = sum log L_jj, info (1 = non-positive pivot,
// 2 = NaN pivot; the first failure of a factorisation wins).  One CTA, latency-bound, so everything is about the
// length of the dependency chain:
//   * each 32x32 diagonal sub-block is factored by one warp in registers, four columns at a time: the 4x4 pivot
//     block is broadcast by shuffle and factored redundantly by every lane, each lane solves its own row against
//     it, and one shared-memory exchange per micro-panel feeds the (unpredicated) rank-4 update; rsqrt + one
//     Newton step replaces sqrt and division (measured on B200: DFMA 8 cycles, rsqrt 74, sqrt 98, div 79);
//   * the rows below a diagonal sub-block are solved by substitution, one lane per row, from the transposed factor;
//   * the SYRK that gates the next sub-block runs as four 8-row strips on warps 0-3 (named barrier 6), the other
//     block pairs on the remaining warps of the main group (named barrier 1, warps 0-6);
//   * warp 7 inverts each sub-block as soon as it is final (named barriers 2..5) by right-looking substitution
//     and stores it; warp 3 streams finished block columns of L out; the off-diagonal blocks of the inverse are
//     assembled in four rounds (T = X_ii L_ik first, then the block columns in parallel).
constexpr int LTLD = 34;                               // transposed-factor row stride (even: 16-byte rows)
constexpr int L2_S = TILE * LLD;                       // S      [128][LLD]
constexpr int L2_XD = TILE;                            // xd     [128]  1/L_jj
constexpr int L2_X = 4 * LB * TLD;                     // Xd     [4][32][TLD] diagonal sub-block inverses (row-major)
constexpr int L2_T = 6 * LB * TLD;                     // T      [6][32][TLD]; aliases LT [4][32][LTLD] while factorising
constexpr int LEAF2_SMEM_BYTES = (L2_S + L2_XD + L2_X + L2_T) * 8;
static_assert(4 * LB * LTLD <= L2_T, "LT must fit in the T region");
static_assert(LEAF2_SMEM_BYTES <= 232448, "leaf v2 shared memory exceeds the 227 KB per-CTA limit");

__device__ __forceinline__ void named_bar_sync(int id, int count) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(count) : "memory");
}
__device__ __forceinline__ void named_bar_arrive(int id, int count) {
    asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(count) : "memory");
}

// One warp: rows row0..row0+31 of the block column b: x <- x * L_bb^-T by substitution (lane = row).
__device__ __forceinline__ void warp_trsm_sub32(double* S, const double* xd, const double* LT, int row0, int b,
                                                int lane) {
    double x[LB];
    double* row = S + (row0 + lane) * LLD + b;
#pragma unroll
    for (int k = 0; k < LB; k += 2) {
        const double2 v = *reinterpret_cast<const double2*>(row + k);
        x[k] = v.x;
        x[k + 1] = v.y;
    }
#pragma unroll
    for (int j = 0; j < LB; j++) {
        x[j] *= xd[b + j];
        const double xj = x[j];
#pragma unroll
        for (int k = (j + 1) & ~1; k < LB; k += 2) {
            const double2 lk = *reinterpret_cast<const double2*>(LT + j * LTLD + k);
            if (k > j) x[k] = fma(-xj, lk.x, x[k]);
            x[k + 1] = fma(-xj, lk.y, x[k + 1]);
        }
    }
#pragma unroll
    for (int k = 0; k < LB; k += 2) {
        double2 v;
        v.x = x[k];
        v.y = x[k + 1];
        *reinterpret_cast<double2*>(row + k) = v;
    }
}

// 32x32 diagonal factorisation by one warp (lane i owns row i), four columns at a time.  The 4x4 pivot block is broadcast by
// shuffle and factored redundantly by every lane (no communication inside the micro-panel), each lane then
// solves its own row against it, and one shared-memory exchange per micro-panel feeds the rank-4 update of the
// remaining columns.  Updates are not predicated: entries above the diagonal hold bounded garbage that is
// never read.  ~1400 instructions per block instead of ~4100, 8 exchanges instead of 32.
#define GPP_PIVOT(d, rs, l)                                       \
    if (!((d) > 0.0) && bad == 0) bad = ((d) != (d)) ? 2 : 1;     \
    rs = rsqrt(d);                                                \
    l = (d) * rs;                                                 \
    l = fma(fma(-l, l, (d)), 0.5 * rs, l);                        \
    rs = fma(fma(-l, rs, 1.0), rs, rs);

__device__ __forceinline__ void warp_potrf32(double* S, double* xd, double* LT, int b, int lane, int& bad,
                                                double& mant, int& esum) {
    double a[LB];
    double* row = S + (b + lane) * LLD + b;
#pragma unroll
    for (int k = 0; k < LB; k += 2) {
        const double2 v = *reinterpret_cast<const double2*>(row + k);
        a[k] = (k <= lane) ? v.x : 0.0;
        a[k + 1] = (k + 1 <= lane) ? v.y : 0.0;
    }
    double mydinv = 0.0;
#pragma unroll
    for (int c0 = 0; c0 < LB; c0 += 4) {
        const double p00 = __shfl_sync(FULL, a[c0], c0);
        const double p10 = __shfl_sync(FULL, a[c0], c0 + 1), p11 = __shfl_sync(FULL, a[c0 + 1], c0 + 1);
        const double p20 = __shfl_sync(FULL, a[c0], c0 + 2), p21 = __shfl_sync(FULL, a[c0 + 1], c0 + 2);
        const double p22 = __shfl_sync(FULL, a[c0 + 2], c0 + 2);
        const double p30 = __shfl_sync(FULL, a[c0], c0 + 3), p31 = __shfl_sync(FULL, a[c0 + 1], c0 + 3);
        const double p32 = __shfl_sync(FULL, a[c0 + 2], c0 + 3), p33 = __shfl_sync(FULL, a[c0 + 3], c0 + 3);
        double r0, r1, r2, r3, l00, l11, l22, l33;
        GPP_PIVOT(p00, r0, l00)
        const double l10 = p10 * r0, l20 = p20 * r0, l30 = p30 * r0;
        const double d1 = fma(-l10, l10, p11);
        GPP_PIVOT(d1, r1, l11)
        const double l21 = fma(-l20, l10, p21) * r1, l31 = fma(-l30, l10, p31) * r1;
        const double d2 = fma(-l21, l21, fma(-l20, l20, p22));
        GPP_PIVOT(d2, r2, l22)
        const double l32 = fma(-l31, l21, fma(-l30, l20, p32)) * r2;
        const double d3 = fma(-l32, l32, fma(-l31, l31, fma(-l30, l30, p33)));
        GPP_PIVOT(d3, r3, l33)
        {
            int ex;
            mant *= frexp((l00 * l11) * (l22 * l33), &ex);
            esum += ex;
        }
        // this lane's row against the pivot block
        double x0 = a[c0] * r0;
        double x1 = fma(-x0, l10, a[c0 + 1]) * r1;
        double x2 = fma(-x1, l21, fma(-x0, l20, a[c0 + 2])) * r2;
        double x3 = fma(-x2, l32, fma(-x1, l31, fma(-x0, l30, a[c0 + 3]))) * r3;
        const int rel = lane - c0;  // rows of the pivot block: exact diagonal, zeros above it; finished rows: zeros
        x0 = (rel == 0) ? l00 : ((rel < 0) ? 0.0 : x0);
        x1 = (rel == 1) ? l11 : ((rel < 1) ? 0.0 : x1);
        x2 = (rel == 2) ? l22 : ((rel < 2) ? 0.0 : x2);
        x3 = (rel == 3) ? l33 : ((rel < 3) ? 0.0 : x3);
        mydinv = (rel == 0) ? r0 : ((rel == 1) ? r1 : ((rel == 2) ? r2 : ((rel == 3) ? r3 : mydinv)));
        a[c0] = x0;
        a[c0 + 1] = x1;
        a[c0 + 2] = x2;
        a[c0 + 3] = x3;
        LT[(c0 + 0) * LTLD + lane] = x0;
        LT[(c0 + 1) * LTLD + lane] = x1;
        LT[(c0 + 2) * LTLD + lane] = x2;
        LT[(c0 + 3) * LTLD + lane] = x3;
        __syncwarp();
#pragma unroll
        for (int j = c0 + 4; j < LB; j += 2) {
            const double2 k0 = *reinterpret_cast<const double2*>(LT + (c0 + 0) * LTLD + j);
            const double2 k1 = *reinterpret_cast<const double2*>(LT + (c0 + 1) * LTLD + j);
            const double2 k2 = *reinterpret_cast<const double2*>(LT + (c0 + 2) * LTLD + j);
            const double2 k3 = *reinterpret_cast<const double2*>(LT + (c0 + 3) * LTLD + j);
            a[j] = fma(-x3, k3.x, fma(-x2, k2.x, fma(-x1, k1.x, fma(-x0, k0.x, a[j]))));
            a[j + 1] = fma(-x3, k3.y, fma(-x2, k2.y, fma(-x1, k1.y, fma(-x0, k0.y, a[j + 1]))));
        }
    }
#pragma unroll
    for (int k = 0; k < LB; k += 2) {
        if (k <= lane) {
            double2 v;
            v.x = a[k];
            v.y = (k + 1 <= lane) ? a[k + 1] : 0.0;
            *reinterpret_cast<double2*>(row + k) = v;
        }
    }
    xd[b + lane] = mydinv;
}
#undef GPP_PIVOT

// rows i0+8w .. i0+8w+7 of the SYRK update of the diagonal sub-block (i0,i0) with block column b (one warp)
__device__ __forceinline__ void warp_syrk_strip8(double* S, int i0, int b, int w, int g, int t) {
    double c[4][2];
#pragma unroll
    for (int ni = 0; ni < 4; ni++) { c[ni][0] = 0.0; c[ni][1] = 0.0; }
#pragma unroll
    for (int kk = 0; kk < LB; kk += 4) {
        const double af = S[(i0 + 8 * w + g) * LLD + b + kk + t];
#pragma unroll
        for (int ni = 0; ni < 4; ni++) {
            if (ni <= w) {
                const double bf = S[(i0 + ni * 8 + g) * LLD + b + kk + t];
                dmma884(c[ni][0], c[ni][1], af, bf);
            }
        }
    }
#pragma unroll
    for (int ni = 0; ni < 4; ni++) {
        if (ni <= w) {
            double2* p2 = reinterpret_cast<double2*>(S + (i0 + 8 * w + g) * LLD + i0 + ni * 8 + 2 * t);
            double2 v = *p2;
            v.x -= c[ni][0];
            v.y -= c[ni][1];
            *p2 = v;
        }
    }
}


// One warp: X = L_bb^-1 by right-looking substitution on the identity (lane c owns column c): the dependent
// chain per row is one multiply and one FMA instead of a half-row dot product.  LT[j][i] = L_ij.
__device__ __forceinline__ void warp_trinv32(const double* LT, const double* xd, double* Xd, int b, int lane) {
    double x[LB];
#pragma unroll
    for (int r = 0; r < LB; r++) x[r] = (r == lane) ? 1.0 : 0.0;
#pragma unroll
    for (int r = 0; r < LB; r++) {
        x[r] *= xd[b + r];
        const double xr = x[r];
#pragma unroll
        for (int k = (r + 1) & ~1; k < LB; k += 2) {
            const double2 lk = *reinterpret_cast<const double2*>(LT + r * LTLD + k);
            if (k > r) x[k] = fma(-xr, lk.x, x[k]);
            x[k + 1] = fma(-xr, lk.y, x[k + 1]);
        }
        Xd[r * TLD + lane] = xr;
    }
}

// One warp: copy rows [r0, r1) x 32 columns of a shared-memory block (leading dimension lds) to global memory
__device__ __forceinline__ void warp_store_rows32(const double* src, int lds, double* dst, long long ldg, int r0,
                                                  int r1, int lane) {
    for (int r = r0; r < r1; r++) dst[(long long)r * ldg + lane] = src[r * lds + lane];
}

__device__ __forceinline__ void acc_store32(double* dst, int ldd, const double (&acc)[4][4][2], double sgn, int g,
                                            int t) {
#pragma unroll
    for (int mi = 0; mi < 4; mi++)
#pragma unroll
        for (int ni = 0; ni < 4; ni++) {
            double2 v;
            v.x = sgn * acc[mi][ni][0];
            v.y = sgn * acc[mi][ni][1];
            *reinterpret_cast<double2*>(dst + (mi * 8 + g) * ldd + ni * 8 + 2 * t) = v;
        }
}

// prof (optional): clock64 stamps written by thread 0 / lane 0 of the inverse warp
__device__ __forceinline__ void leaf_potrf_trinv_body(double* A, int ld, int kb, double* M, double* logdet_part, int* info,
                                                      long long* prof, double* sm) {
    double* S = sm;
    double* xd = S + L2_S;
    double* Xd = xd + L2_XD;
    double* Tr = Xd + L2_X;
    double* LT = Tr;  // alias: only used while factorising
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int g = lane >> 2, t = lane & 3;
    double* Ab = A + (long long)kb * TILE * ld + (long long)kb * TILE;
    double* Mb = M + (long long)kb * TILE * ld + (long long)kb * TILE;
#define GPP_STAMP(i) \
    if (prof && tid == 0) prof[i] = clock64();

    GPP_STAMP(0)
    // whole rows with 16-byte loads (the strict upper part is never read by the factorisation)
    for (int idx = tid; idx < TILE * (TILE / 2); idx += LEAF_THREADS) {
        const int i = idx >> 6, j2 = (idx & 63) * 2;
        if (j2 <= i)
            *reinterpret_cast<double2*>(S + i * LLD + j2) = *reinterpret_cast<const double2*>(Ab + (long long)i * ld + j2);
    }
    __syncthreads();
    GPP_STAMP(1)

    double acc[4][4][2];
    if (warp == 7) {
        // inverse warp: X_qq as soon as L_qq is final
        for (int q = 0; q < 4; q++) {
            named_bar_sync(2 + q, 64);
            warp_trinv32(LT + q * LB * LTLD, xd, Xd + q * LB * TLD, q * LB, lane);
            __syncwarp();
            // the diagonal sub-block of the inverse is final: store it now, off the tail
            warp_store_rows32(Xd + q * LB * TLD, TLD, Mb + (long long)(q * LB) * ld + q * LB, ld, 0, LB, lane);
        }
        if (prof && lane == 0) prof[15] = clock64();
    } else {
        int bad = 0, esum = 0;
        double mant = 1.0;
        for (int q = 0; q < 4; q++) {
            const int b = q * LB;
            if (warp == 0) {
                warp_potrf32(S, xd, LT + q * LB * LTLD, b, lane, bad, mant, esum);
                __threadfence_block();
                named_bar_arrive(2 + q, 64);
            }
            GPP_STAMP(2 + 3 * q)
            if (q == 3) break;
            named_bar_sync(1, 224);
            if (warp >= 1 && warp <= 3 - q) warp_trsm_sub32(S, xd, LT + q * LB * LTLD, (q + warp) * LB, b, lane);
            named_bar_sync(1, 224);
            GPP_STAMP(3 + 3 * q)
            {
                // SYRK: the next diagonal block (it gates the next factorisation) in four 8-row strips on warps 0-3,
                // the other block pairs on warps 4,5,6,1,2 in that order
                const int i0d = (q + 1) * LB;
                if (warp < 4) {
                    warp_syrk_strip8(S, i0d, b, warp, g, t);
                    named_bar_sync(6, 128);
                }
                if (warp == 3) {
                    // block column q of L is final (diagonal sub-block after the factorisation, the rows below it
                    // after the substitution): stream it out while the other warps update the trailing blocks
                    for (int r = b; r < TILE; r++) {
                        const int c = b + lane;
                        if (c <= r) Ab[(long long)r * ld + c] = S[r * LLD + c];
                    }
                }
                const int m = 3 - q;
                const int npairs = m * (m + 1) / 2 - 1;
                const int slot = (warp >= 4) ? warp - 4 : (warp >= 1 ? warp + 2 : -1);  // warps 4,5,6,1,2,3 -> 0..5
                if (slot >= 0 && slot < npairs) {
                    int u = 0, w = slot + 1;  // pair index slot+1 in the (u,w) enumeration, pair 0 is the diagonal
                    while (w > u) { w -= u + 1; u++; }
                    const int i0 = (q + 1 + u) * LB, j0 = (q + 1 + w) * LB;
                    acc_zero(acc);
                    warp_mm32(acc, [&](int r, int k) { return S[(i0 + r) * LLD + b + k]; },
                              [&](int k, int c) { return S[(j0 + c) * LLD + b + k]; }, g, t);
#pragma unroll
                    for (int mi = 0; mi < 4; mi++)
#pragma unroll
                        for (int ni = 0; ni < 4; ni++) {
                            const int r = mi * 8 + g, c = ni * 8 + 2 * t;
                            double2* p2 = reinterpret_cast<double2*>(S + (i0 + r) * LLD + j0 + c);
                            double2 v = *p2;
                            v.x -= acc[mi][ni][0];
                            v.y -= acc[mi][ni][1];
                            *p2 = v;
                        }
                }
            }
            GPP_STAMP(4 + 3 * q)
        }
        if (warp == 0 && lane == 0) {
            logdet_part[kb] = log(mant) + (double)esum * 0.6931471805599453;
            if (bad && *info == 0) atomicOr(info, bad);  // leaves run in sequence: an earlier failure wins
        }
    }
    __syncthreads();
    GPP_STAMP(14)

    // ---- off-diagonal 32-blocks of X = L^-1.  X_ij (i > j) is kept row-major in the unused block (j,i) of S. ----
    // round 0: T_ik = X_ii L_ik, six blocks
    if (warp < 6) {
        int i = 1, k = warp;
        while (k >= i) { k -= i; i++; }  // warp -> (i,k): (1,0) (2,0) (2,1) (3,0) (3,1) (3,2)
        acc_zero(acc);
        const double* Xi = Xd + i * LB * TLD;
        warp_mm32(acc, [&](int r, int kk) { return Xi[r * TLD + kk]; },
                  [&](int kk, int n) { return S[(i * LB + kk) * LLD + k * LB + n]; }, g, t);
        acc_store32(Tr + warp * LB * TLD, TLD, acc, 1.0, g, t);
    }
    __syncthreads();
    // T index of (i,k): i(i-1)/2 + k
#define GPP_T(i, k) (Tr + ((i) * ((i) - 1) / 2 + (k)) * LB * TLD)
#define GPP_XOFF(i, j) (S + ((j) * LB) * LLD + (i) * LB)  // row-major container of X_ij, leading dimension LLD
    // round 1: X_10, X_21, X_32 (stored) and the first terms of X_20, X_31, X_30 (kept in registers)
    if (warp < 6) {
        // warps 0..2: (i,j) = (1,0) (2,1) (3,2);  warps 3..5: (2,0) (3,1) (3,0)
        const int i = (warp < 3) ? warp + 1 : (warp == 3 ? 2 : 3);
        const int j = (warp < 3) ? warp : (warp == 5 ? 0 : warp - 3);
        acc_zero(acc);
        const double* Tij = GPP_T(i, j);
        const double* Xj = Xd + j * LB * TLD;
        warp_mm32(acc, [&](int r, int kk) { return Tij[r * TLD + kk]; },
                  [&](int kk, int n) { return Xj[kk * TLD + n]; }, g, t);
        if (warp < 3) acc_store32(GPP_XOFF(i, j), LLD, acc, -1.0, g, t);
    }
    __syncthreads();
    // round 2: X_20 = -(P_20 + T_21 X_10) [warp 3], X_31 = -(P_31 + T_32 X_21) [warp 4], P_30 += T_31 X_10 [warp 5]
    if (warp >= 3 && warp < 6) {
        const int i = (warp == 3) ? 2 : 3;
        const int j = (warp == 4) ? 1 : 0;
        const int k = j + 1;
        const double* Tik = GPP_T(i, k);
        const double* Xkj = GPP_XOFF(k, j);
        warp_mm32(acc, [&](int r, int kk) { return Tik[r * TLD + kk]; },
                  [&](int kk, int n) { return Xkj[kk * LLD + n]; }, g, t);
        if (warp < 5) acc_store32(GPP_XOFF(i, j), LLD, acc, -1.0, g, t);
    }
    __syncthreads();
    // round 3: X_30 = -(P_30 + T_32 X_20) [warp 5]
    if (warp == 5) {
        const double* Tik = GPP_T(3, 2);
        const double* Xkj = GPP_XOFF(2, 0);
        warp_mm32(acc, [&](int r, int kk) { return Tik[r * TLD + kk]; },
                  [&](int kk, int n) { return Xkj[kk * LLD + n]; }, g, t);
        acc_store32(GPP_XOFF(3, 0), LLD, acc, -1.0, g, t);
    }
    __syncthreads();
    GPP_STAMP(12)
#undef GPP_T

    {
        // everything except the last diagonal sub-block of L and the six off-diagonal sub-blocks of the inverse
        // has already been stored; 7 block copies over 8 warps
        if (warp == 7) {
            for (int r = 3 * LB; r < TILE; r++) {
                const int c = 3 * LB + lane;
                if (c <= r) Ab[(long long)r * ld + c] = S[r * LLD + c];
            }
        } else if (warp < 6) {
            int i = 1, j = warp;
            while (j >= i) { j -= i; i++; }  // warp -> (i,j): (1,0) (2,0) (2,1) (3,0) (3,1) (3,2)
            warp_store_rows32(GPP_XOFF(i, j), LLD, Mb + (long long)(i * LB) * ld + j * LB, ld, 0, LB, lane);
        }
    }
#undef GPP_XOFF
    GPP_STAMP(13)
#undef GPP_STAMP
}

__global__ void __launch_bounds__(LEAF_THREADS, 1)
leaf_potrf_trinv_kernel(double* A, int ld, int kb, double* M, double* logdet_part, int* info, long long* prof) {
    extern __shared__ __align__(16) double sm[];
    leaf_potrf_trinv_body(A, ld, kb, M, logdet_part, info, prof, sm);
}

// ---------------------------------------------------------------------------------------------
// Diagonal block of a panel (pw x pw tiles, pw <= 16) in ONE launch: a left-looking tile dataflow.  The tiles are
// numbered column by column; CTA c handles tiles c, c + G, c + 2G, ... in that order.  Tile (i,j), i > j:
//   P = sum_{k<j} L(i,k) L(j,k)^T (DMMA, operands streamed from L2 as soon as their flags are up),
//   L(i,j) = (A(i,j) - P) L_jj^-T   via the explicit inverse of the diagonal tile (as the TRSM launches do);
// tile (j,j): A(j,j) -= sum_{k<j} L(j,k) L(j,k)^T, then the leaf (factor + inverse) in place.
// A finished tile is published with a release store of the launch's epoch to its flag; consumers spin on an acquire
// load.  Dependencies only point to lower tile numbers and CTAs are dispatched in index order, so the scheme cannot
// deadlock even when only some CTAs are resident.  Replaces ~37 dependent launches per 12-tile block
// (leaf / TRSM / update / recursion updates: ~135 us per 128-column step) by flag hand-offs (~75 us per step).
constexpr int BLKP_THREADS = 256;
constexpr int BLKP_NST = 3;
constexpr int BLKP_XLD = 132;
constexpr int BLKP_STAGE = TILE * LDS_KC;   // doubles per operand and stage
constexpr int BLKP_SMEM_TRSM = (TILE * BLKP_XLD + BLKP_NST * BLKP_STAGE) * 8;
constexpr int BLKP_SMEM_UPD = (2 * BLKP_NST * BLKP_STAGE) * 8;
constexpr int BLKP_SMEM_BYTES = (LEAF2_SMEM_BYTES > BLKP_SMEM_TRSM ? LEAF2_SMEM_BYTES : BLKP_SMEM_TRSM) > BLKP_SMEM_UPD
                                    ? (LEAF2_SMEM_BYTES > BLKP_SMEM_TRSM ? LEAF2_SMEM_BYTES : BLKP_SMEM_TRSM)
                                    : BLKP_SMEM_UPD;
static_assert(BLKP_SMEM_BYTES <= 232448, "block factorisation shared memory exceeds the 227 KB per-CTA limit");
static_assert(LEAF_THREADS == BLKP_THREADS, "the leaf body runs inside the block kernel");

__device__ __forceinline__ void blkp_wait(const int* flag, int epoch) {
    if (threadIdx.x == 0) {
        int v;
        unsigned spins = 0;
        for (;;) {
            asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(flag) : "memory");
            if (v == epoch) break;
            __nanosleep(100);
            if (++spins > (1u << 24)) __trap();   // ~2 s: a lost hand-off surfaces as a CUDA error, not a hang
        }
    }
    __syncthreads();
}
__device__ __forceinline__ void blkp_post(int* flag, int epoch) {
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(flag), "r"(epoch) : "memory");
}

// acc += A(128 x 128) B(128 x 128)^T, both operands k-contiguous in global memory (read through L2 by cp.async.cg)
__device__ __forceinline__ void blkp_mma_gg(double (&acc)[4][8][2], const double* Ag, int lda, const double* Bg, int ldb,
                                            double* pipe, int tid, int wm0, int wn0, int g, int t) {
    constexpr int NCH = TILE / BK;
    double* sA = pipe;
    double* sB = pipe + BLKP_NST * BLKP_STAGE;
#pragma unroll
    for (int s = 0; s < BLKP_NST - 1; s++) {
        load_chunk<true, TILE, BLKP_THREADS>(sA + s * BLKP_STAGE, Ag + s * BK, lda, tid);
        load_chunk<true, TILE, BLKP_THREADS>(sB + s * BLKP_STAGE, Bg + s * BK, ldb, tid);
        cp_async_commit();
    }
    for (int c = 0; c < NCH; c++) {
        cp_async_wait<BLKP_NST - 2>();
        __syncthreads();
        const int cn = c + BLKP_NST - 1;
        if (cn < NCH) {
            const int s = cn % BLKP_NST;
            load_chunk<true, TILE, BLKP_THREADS>(sA + s * BLKP_STAGE, Ag + cn * BK, lda, tid);
            load_chunk<true, TILE, BLKP_THREADS>(sB + s * BLKP_STAGE, Bg + cn * BK, ldb, tid);
        }
        cp_async_commit();
        const double* a_s = sA + (c % BLKP_NST) * BLKP_STAGE;
        const double* b_s = sB + (c % BLKP_NST) * BLKP_STAGE;
#pragma unroll
        for (int kk = 0; kk < BK / 4; kk++) {
            double af[4], bf[8];
#pragma unroll
            for (int mi = 0; mi < 4; mi++) af[mi] = a_s[(wm0 + mi * 8 + g) * LDS_KC + kk * 4 + t];
#pragma unroll
            for (int ni = 0; ni < 8; ni++) bf[ni] = b_s[(wn0 + ni * 8 + g) * LDS_KC + kk * 4 + t];
#pragma unroll
            for (int mi = 0; mi < 4; mi++)
#pragma unroll
                for (int ni = 0; ni < 8; ni++) dmma884(acc[mi][ni][0], acc[mi][ni][1], af[mi], bf[ni]);
        }
    }
    cp_async_wait<0>();
    __syncthreads();
}

// acc = Xs(128 x 128, shared memory, leading dimension BLKP_XLD) B(128 x 128)^T, B k-contiguous in global memory
__device__ __forceinline__ void blkp_mma_sg(double (&acc)[4][8][2], const double* Xs, const double* Bg, int ldb, double* pipe,
                                            int tid, int wm0, int wn0, int g, int t) {
    constexpr int NCH = TILE / BK;
    double* sB = pipe;
#pragma unroll
    for (int s = 0; s < BLKP_NST - 1; s++) {
        load_chunk<true, TILE, BLKP_THREADS>(sB + s * BLKP_STAGE, Bg + s * BK, ldb, tid);
        cp_async_commit();
    }
    for (int c = 0; c < NCH; c++) {
        cp_async_wait<BLKP_NST - 2>();
        __syncthreads();
        const int cn = c + BLKP_NST - 1;
        if (cn < NCH) load_chunk<true, TILE, BLKP_THREADS>(sB + (cn % BLKP_NST) * BLKP_STAGE, Bg + cn * BK, ldb, tid);
        cp_async_commit();
        const double* b_s = sB + (c % BLKP_NST) * BLKP_STAGE;
#pragma unroll
        for (int kk = 0; kk < BK / 4; kk++) {
            double af[4], bf[8];
#pragma unroll
            for (int mi = 0; mi < 4; mi++) af[mi] = Xs[(wm0 + mi * 8 + g) * BLKP_XLD + c * BK + kk * 4 + t];
#pragma unroll
            for (int ni = 0; ni < 8; ni++) bf[ni] = b_s[(wn0 + ni * 8 + g) * LDS_KC + kk * 4 + t];
#pragma unroll
            for (int mi = 0; mi < 4; mi++)
#pragma unroll
                for (int ni = 0; ni < 8; ni++) dmma884(acc[mi][ni][0], acc[mi][ni][1], af[mi], bf[ni]);
        }
    }
    cp_async_wait<0>();
    __syncthreads();
}

struct BlockPotrfArgs {
    double* A;            // whole matrix (leading dimension ld)
    double* M;
    int ld;
    int t0, pw;           // first tile and width of the diagonal block
    double* logdet_part;
    int* info;
    int* flags;           // [pw * pw], value == epoch: tile final
    int epoch;
};

__global__ void __launch_bounds__(BLKP_THREADS, 1) block_potrf_kernel(const BlockPotrfArgs a) {
    extern __shared__ __align__(16) double sm[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int g = lane >> 2, t = lane & 3;
    const int wm0 = (warp >> 1) * 32, wn0 = (warp & 1) * 64;
    const int pw = a.pw, ld = a.ld;
    const int ntiles = pw * (pw + 1) / 2;
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        // column-major numbering of the lower tiles: column j holds rows j .. pw-1
        int j = 0, rem = tile;
        while (rem >= pw - j) { rem -= pw - j; j++; }
        const int i = j + rem;
        double* Aij = a.A + (long long)(a.t0 + i) * TILE * ld + (long long)(a.t0 + j) * TILE;
        double acc[4][8][2];
#pragma unroll
        for (int mi = 0; mi < 4; mi++)
#pragma unroll
            for (int ni = 0; ni < 8; ni++) { acc[mi][ni][0] = 0.0; acc[mi][ni][1] = 0.0; }
        for (int k = 0; k < j; k++) {
            blkp_wait(a.flags + i * pw + k, a.epoch);
            if (i != j) blkp_wait(a.flags + j * pw + k, a.epoch);
            const double* Lik = a.A + (long long)(a.t0 + i) * TILE * ld + (long long)(a.t0 + k) * TILE;
            const double* Ljk = a.A + (long long)(a.t0 + j) * TILE * ld + (long long)(a.t0 + k) * TILE;
            blkp_mma_gg(acc, Lik, ld, Ljk, ld, sm, tid, wm0, wn0, g, t);
        }
        if (i == j) {
            // updated diagonal tile back to global memory, then factor + invert it in place
            if (j > 0) {
#pragma unroll
                for (int mi = 0; mi < 4; mi++)
#pragma unroll
                    for (int ni = 0; ni < 8; ni++) {
                        double2* p2 = reinterpret_cast<double2*>(Aij + (long long)(wm0 + mi * 8 + g) * ld + wn0 + ni * 8 + 2 * t);
                        double2 v = *p2;
                        v.x -= acc[mi][ni][0];
                        v.y -= acc[mi][ni][1];
                        *p2 = v;
                    }
                __threadfence();
                __syncthreads();
            }
            leaf_potrf_trinv_body(a.A, ld, a.t0 + j, a.M, a.logdet_part, a.info, nullptr, sm);
            blkp_post(a.flags + j * pw + j, a.epoch);
        } else {
            // X = A(i,j) - P into shared memory, then L(i,j) = X L_jj^-T
            double* Xs = sm;
            double* pipe = sm + TILE * BLKP_XLD;
#pragma unroll
            for (int mi = 0; mi < 4; mi++)
#pragma unroll
                for (int ni = 0; ni < 8; ni++) {
                    const int r = wm0 + mi * 8 + g, c = wn0 + ni * 8 + 2 * t;
                    double2 v = *reinterpret_cast<const double2*>(Aij + (long long)r * ld + c);
                    v.x -= acc[mi][ni][0];
                    v.y -= acc[mi][ni][1];
                    *reinterpret_cast<double2*>(Xs + r * BLKP_XLD + c) = v;
                    acc[mi][ni][0] = 0.0;
                    acc[mi][ni][1] = 0.0;
                }
            blkp_wait(a.flags + j * pw + j, a.epoch);   // L_jj^-1 is in M (also orders the Xs stores before the reads)
            const double* Winv = a.M + (long long)(a.t0 + j) * TILE * ld + (long long)(a.t0 + j) * TILE;
            blkp_mma_sg(acc, Xs, Winv, ld, pipe, tid, wm0, wn0, g, t);
#pragma unroll
            for (int mi = 0; mi < 4; mi++)
#pragma unroll
                for (int ni = 0; ni < 8; ni++) {
                    double2 v;
                    v.x = acc[mi][ni][0];
                    v.y = acc[mi][ni][1];
                    *reinterpret_cast<double2*>(Aij + (long long)(wm0 + mi * 8 + g) * ld + wn0 + ni * 8 + 2 * t) = v;
                }
            blkp_post(a.flags + i * pw + j, a.epoch);
        }
        __syncthreads();   // shared memory is re-carved by the next tile
    }
}

inline cudaError_t chol_set_attributes() {
    cudaError_t e = cudaFuncSetAttribute(leaf_potrf_trinv_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         LEAF2_SMEM_BYTES);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(block_potrf_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, BLKP_SMEM_BYTES);
    if (e != cudaSuccess) return e;
    e = oz_set_attributes();
    if (e != cudaSuccess) return e;
    return gemm_set_attributes();
}

// diagonal block [t0, t0 + pw) of A in one launch (flags: pw * pw ints owned by the caller; epoch must differ from every
// value left in them, e.g. a per-handle launch counter)
inline cudaError_t launch_block_potrf(double* A, double* M, int ld, int t0, int pw, double* logdet_part, int* info, int* flags,
                                      int epoch, int ctas, cudaStream_t st) {
    BlockPotrfArgs a;
    a.A = A;
    a.M = M;
    a.ld = ld;
    a.t0 = t0;
    a.pw = pw;
    a.logdet_part = logdet_part;
    a.info = info;
    a.flags = flags;
    a.epoch = epoch;
    const int ntiles = pw * (pw + 1) / 2;
    const int gx = ctas < ntiles ? ctas : ntiles;
    block_potrf_kernel<<<gx, BLKP_THREADS, BLKP_SMEM_BYTES, st>>>(a);
    count_launch();
    return cudaGetLastError();
}

inline cudaError_t launch_leaf(double* A, int ld, int col, double* M, double* logdet_part, int* info, cudaStream_t st,
                               long long* prof = nullptr) {
    leaf_potrf_trinv_kernel<<<1, LEAF_THREADS, LEAF2_SMEM_BYTES, st>>>(A, ld, col, M, logdet_part, info, prof);
    count_launch();
    return cudaGetLastError();
}

#define GPP_TRY(x)                      \
    do {                                \
        cudaError_t _e = (x);           \
        if (_e != cudaSuccess) return _e; \
    } while (0)

// A (lower) -> L in place; diagonal blocks of M <- inverse of the diagonal blocks of L.
inline cudaError_t potrf_blocked(double* A, double* M, int ld, int T, double* logdet_part, int* info,
                                 cudaStream_t st) {
    for (int p0 = 0; p0 < T; p0 += PANEL_BLOCKS) {
        const int pw = (T - p0 < PANEL_BLOCKS) ? (T - p0) : PANEL_BLOCKS;
        const int pend = p0 + pw;
        for (int col = p0; col < pend; col++) {
            GPP_TRY(launch_leaf(A, ld, col, M, logdet_part, info, st));
            const int below = T - col - 1;
            if (below <= 0) continue;
            {   // TRSM: A[i,col] <- A[i,col] * Linv_col^T   (in place; a CTA only reads its own rows)
                GemmOp op = gemm_default();
                op.A = A + (long long)(col + 1) * TILE * ld + (long long)col * TILE;
                op.lda = ld;
                op.B = M + (long long)col * TILE * ld + (long long)col * TILE;
                op.ldb = ld;
                op.C = const_cast<double*>(op.A);
                op.ldc = ld;
                op.tiles_m = op.tiles_m_last = below;
                op.tiles_n = 1;
                op.klo_c = 0;
                op.khi_c = 1;
                GPP_TRY(launch_gemm(op, true, true, 1, st));
            }
            const int pc = pend - col - 1;  // panel columns still to update
            if (pc > 0) {
                // A[i,j] -= A[i,col] * A[j,col]^T  for col < j < pend, i >= j
                GemmOp op = gemm_default();
                op.A = A + (long long)(col + 1) * TILE * ld + (long long)col * TILE;
                op.lda = ld;
                op.B = op.A;
                op.ldb = ld;
                op.C = A + (long long)(col + 1) * TILE * ld + (long long)(col + 1) * TILE;
                op.ldc = ld;
                op.tiles_m = op.tiles_m_last = below;
                op.tiles_n = pc;
                op.lower_filter = 1;
                op.lower_off = 0;
                op.klo_c = 0;
                op.khi_c = 1;
                op.alpha = -1.0;
                op.beta = 1.0;
                GPP_TRY(launch_gemm(op, true, true, 1, st));
            }
        }
        const int rest = T - pend;
        if (rest > 0) {
            // trailing SYRK: A[i,j] -= sum_{k in panel} A[i,k] A[j,k]^T , i >= j >= pend
            GemmOp op = gemm_default();
            op.A = A + (long long)pend * TILE * ld + (long long)p0 * TILE;
            op.lda = ld;
            op.B = op.A;
            op.ldb = ld;
            op.C = A + (long long)pend * TILE * ld + (long long)pend * TILE;
            op.ldc = ld;
            op.map = MAP_TRI;
            op.tiles_m = op.tiles_m_last = rest;
            op.tiles_n = rest;
            op.klo_c = 0;
            op.khi_c = pw;
            op.alpha = -1.0;
            op.beta = 1.0;
            GPP_TRY(launch_gemm(op, true, true, 1, st));
        }
    }
    return cudaSuccess;
}

// ---------------------------------------------------------------------------------------------
// Look-ahead variant.  The panel factorisation (leaf / TRSM / in-panel update: a chain of small, latency-bound
// launches) runs on a high-priority side stream and overlaps the bulk of the previous panel's trailing update,
// which stays on the main stream:
//
//   side:  PF(0) . TUn(0) PF(1) . [wait TUr(0)] TUn(1) PF(2) . [wait TUr(1)] TUn(2) ...
//   main:        [wait PF(0)] TUr(0)            [wait PF(1)] TUr(1) ...
//
// PF(p)  = factor panel p;  TUn(p) = update of the NEXT panel's tile columns with panel p (rect + lower filter);
// TUr(p) = update of everything to the right of the next panel (lower tiles, the O(N^3) part).
struct CholLookahead {
    cudaStream_t side = nullptr;
    cudaStream_t inv = nullptr;   // lowest priority: early part of the triangular inverse, fills idle SMs
    cudaEvent_t fork = nullptr, join = nullptr, inv_done = nullptr;
    bool inv_pending = false;
    std::vector<cudaEvent_t> ev_pf, ev_tu, ev_m1, ev_s1;
    int panels = 0;

    int* blk_flags = nullptr;   // tile flags of block_potrf_kernel (256 ints), epoch = launch counter
    int blk_epoch = 0;
    int blk_ctas = 24;          // CTAs of one diagonal-block launch (GPP_BLOCK_CTAS; 0 = the launch-per-step chain)
    bool timeline = false;   // GPP_TIMELINE=1 (development): timing-enabled panel events, dumped by dump_timeline()
    cudaError_t init(int T) {
        timeline = getenv("GPP_TIMELINE") != nullptr && atoi(getenv("GPP_TIMELINE")) != 0;
        const unsigned evf = timeline ? cudaEventDefault : cudaEventDisableTiming;
        int lo = 0, hi = 0;
        GPP_TRY(cudaDeviceGetStreamPriorityRange(&lo, &hi));
        GPP_TRY(cudaStreamCreateWithPriority(&side, cudaStreamNonBlocking, hi));
        GPP_TRY(cudaStreamCreateWithPriority(&inv, cudaStreamNonBlocking, lo));
        GPP_TRY(cudaEventCreateWithFlags(&fork, evf));
        GPP_TRY(cudaEventCreateWithFlags(&join, cudaEventDisableTiming));
        GPP_TRY(cudaEventCreateWithFlags(&inv_done, cudaEventDisableTiming));
        GPP_TRY(cudaMalloc(&blk_flags, 256 * sizeof(int)));
        GPP_TRY(cudaMemset(blk_flags, 0, 256 * sizeof(int)));
        if (getenv("GPP_BLOCK_CTAS")) blk_ctas = atoi(getenv("GPP_BLOCK_CTAS"));
        // one set of panel events per tile column: enough for every panel width the schedules accept (GPP_PANEL,
        // GPP_OZ_LAZY_PB down to 2; sizing by PANEL_BLOCKS made narrower panels fail with cudaErrorInvalidValue)
        panels = T;
        ev_pf.resize(panels);
        ev_tu.resize(panels);
        ev_m1.resize(panels);
        ev_s1.resize(panels);
        for (int i = 0; i < panels; i++) {
            GPP_TRY(cudaEventCreateWithFlags(&ev_pf[i], evf));
            GPP_TRY(cudaEventCreateWithFlags(&ev_tu[i], evf));
            GPP_TRY(cudaEventCreateWithFlags(&ev_m1[i], evf));
            GPP_TRY(cudaEventCreateWithFlags(&ev_s1[i], evf));
        }
        return cudaSuccess;
    }
    // ms since the fork of the last factorisation at which each panel event completed (call after a synchronise)
    void dump_timeline(int np) const {
        if (!timeline) return;
        for (int p = 0; p < np && p < panels; p++) {
            float a = -1.f, b = -1.f, c = -1.f, d = -1.f;
            if (cudaEventElapsedTime(&a, fork, ev_pf[p]) != cudaSuccess) a = -1.f;
            if (cudaEventElapsedTime(&b, fork, ev_s1[p]) != cudaSuccess) b = -1.f;
            if (cudaEventElapsedTime(&c, fork, ev_m1[p]) != cudaSuccess) c = -1.f;
            if (cudaEventElapsedTime(&d, fork, ev_tu[p]) != cudaSuccess) d = -1.f;
            fprintf(stderr, "[timeline] panel %2d: block/panel factored %7.3f  s1 %7.3f  m1 %7.3f  m2 %7.3f ms\n", p, a, b, c, d);
        }
        cudaGetLastError();
    }
    void destroy() {
        for (auto e : ev_pf) cudaEventDestroy(e);
        for (auto e : ev_tu) cudaEventDestroy(e);
        for (auto e : ev_m1) cudaEventDestroy(e);
        for (auto e : ev_s1) cudaEventDestroy(e);
        ev_pf.clear();
        ev_tu.clear();
        ev_m1.clear();
        ev_s1.clear();
        if (blk_flags) cudaFree(blk_flags);
        blk_flags = nullptr;
        if (fork) cudaEventDestroy(fork);
        if (join) cudaEventDestroy(join);
        if (inv_done) cudaEventDestroy(inv_done);
        if (side) cudaStreamDestroy(side);
        if (inv) cudaStreamDestroy(inv);
        fork = join = inv_done = nullptr;
        side = inv = nullptr;
    }
};

// factor tile columns [p0, pend) of the panel on stream st (rows p0..T)
inline cudaError_t panel_factor_base(double* A, double* M, int ld, int T, int p0, int pend, double* logdet_part,
                                     int* info, cudaStream_t st) {
    for (int col = p0; col < pend; col++) {
        GPP_TRY(launch_leaf(A, ld, col, M, logdet_part, info, st));
        const int below = T - col - 1;
        if (below <= 0) continue;
        {   // TRSM: A[i,col] <- A[i,col] * Linv_col^T   (in place; a CTA only reads its own rows)
            GemmOp op = gemm_default();
            op.A = A + (long long)(col + 1) * TILE * ld + (long long)col * TILE;
            op.lda = ld;
            op.B = M + (long long)col * TILE * ld + (long long)col * TILE;
            op.ldb = ld;
            op.C = const_cast<double*>(op.A);
            op.ldc = ld;
            op.tiles_m = op.tiles_m_last = below;
            op.tiles_n = 1;
            op.klo_c = 0;
            op.khi_c = 1;
            GPP_TRY(launch_gemm(op, true, true, 1, st));
        }
        const int pc = pend - col - 1;  // panel columns still to update
        if (pc > 0) {
            GemmOp op = gemm_default();
            op.A = A + (long long)(col + 1) * TILE * ld + (long long)col * TILE;
            op.lda = ld;
            op.B = op.A;
            op.ldb = ld;
            op.C = A + (long long)(col + 1) * TILE * ld + (long long)(col + 1) * TILE;
            op.ldc = ld;
            op.tiles_m = op.tiles_m_last = below;
            op.tiles_n = pc;
            op.lower_filter = 1;
            op.lower_off = 0;
            op.klo_c = 0;
            op.khi_c = 1;
            op.alpha = -1.0;
            op.beta = 1.0;
            GPP_TRY(launch_gemm(op, true, true, 1, st));
        }
    }
    return cudaSuccess;
}

// C[i,j] -= sum_{k in [p0,pend)} A[i,k] A[j,k]^T for tile rows i >= r0, tile columns j in [c0, c1), i >= j
inline cudaError_t trailing_update(double* A, int ld, int T, int p0, int pend, int c0, int c1, cudaStream_t st,
                                   int max_ctas = 0) {
    if (c1 <= c0 || c0 >= T) return cudaSuccess;
    GemmOp op = gemm_default();
    op.max_ctas = max_ctas;
    op.A = A + (long long)c0 * TILE * ld + (long long)p0 * TILE;
    op.lda = ld;
    op.B = op.A;
    op.ldb = ld;
    op.C = A + (long long)c0 * TILE * ld + (long long)c0 * TILE;
    op.ldc = ld;
    op.tiles_m = op.tiles_m_last = T - c0;
    op.klo_c = 0;
    op.khi_c = pend - p0;
    op.alpha = -1.0;
    op.beta = 1.0;
    if (c1 >= T) {
        op.map = MAP_TRI;
        op.tiles_n = T - c0;
    } else {
        op.tiles_n = c1 - c0;
        op.lower_filter = 1;
        op.lower_off = 0;
    }
    return launch_gemm(op, true, true, 1, st);
}

// panels wider than PANEL_BLOCKS are factored recursively: left half, update of the right half with the left
// (one DMMA GEMM at K = width/2), right half -- so that only PANEL_BLOCKS-wide pieces run at K = 128
inline cudaError_t panel_factor(double* A, double* M, int ld, int T, int p0, int pend, double* logdet_part, int* info,
                                cudaStream_t st, OzCtx* oz = nullptr) {
    const int w = pend - p0;
    if (w <= PANEL_BASE) return panel_factor_base(A, M, ld, T, p0, pend, logdet_part, info, st);
    int half = PANEL_BASE;
    while (half * 2 < w) half *= 2;
    const int mid = p0 + half;
    GPP_TRY(panel_factor(A, M, ld, T, p0, mid, logdet_part, info, st, oz));
    if (oz && oz->ready && oz->inner_min_k > 0 && half >= oz->inner_min_k && oz_use_trailing(oz, T, mid)) {
        // wide in-panel update on the INT8-sliced GEMM (planes of the left half, rows mid..T; scale slot 4)
        GPP_TRY(oz_split_panel(*oz, A, ld, T, p0, mid, mid, 4, st));
        GPP_TRY(oz_trailing_update(*oz, A, ld, T, p0, mid, mid, pend, 4, st));
    } else {
        GPP_TRY(trailing_update(A, ld, T, p0, mid, mid, pend, st));
    }
    return panel_factor(A, M, ld, T, mid, pend, logdet_part, info, st, oz);
}

inline int g_lookahead_depth = 2;  // 1: the next panel waits for the whole previous trailing update; 2: see below

inline int g_overlap_inverse = 1;   // start the early part of L^-1 (trtri_early) as soon as its columns of L are final

// defined below; X is the scratch of the triangular inverse (may be null: no overlap)
inline int trtri_split_point(int T);

inline cudaError_t trtri_early(const double* L, double* M, double* X, int ld, int T, cudaStream_t st, OzCtx* oz);

inline cudaError_t potrf_lookahead(double* A, double* M, int ld, int T, double* logdet_part, int* info,
                                   cudaStream_t st, CholLookahead& la, double* X = nullptr, OzCtx* oz = nullptr) {
    // K of the trailing update: wide panels only pay off when the trailing matrix is large (measured:
    // N = 16384 59.0 -> 56.6 ms with 8, N = 8192 12.3 -> 12.8 ms; round 2, whole evaluation at N = 16384:
    // 139.3 ms with 8, 138.4 with 12, 138.6 with 16)
    const int PB = g_panel_blocks > 0 ? g_panel_blocks : (T >= 96 ? 12 : 4);
    const int NP = (T + PB - 1) / PB;
    if (NP > la.panels) return cudaErrorInvalidValue;
    const bool deep = g_lookahead_depth >= 2;
    const int H = trtri_split_point(T);
    const bool overlap = g_overlap_inverse && X != nullptr && H > 0 && NP > 1;
    la.inv_pending = false;
    GPP_TRY(cudaEventRecord(la.fork, st));
    GPP_TRY(cudaStreamWaitEvent(la.side, la.fork, 0));
    // Depth-2 schedule.  U(p,c) = update of panel c's tile columns with panel p.
    //   side:  PF(0) U(0,1) PF(1) [wait U(0,2)] U(1,2) PF(2) [wait U(1,3)] U(2,3) ...
    //   main:  [wait PF(0)] U(0,2) U(0,3..) [wait PF(1)] U(1,3) U(1,4..) ...
    // The side chain only waits for U(p-1,p+1), which the main stream issues BEFORE the bulk U(p-1,p+2..), so it can
    // run one panel further ahead than with a single trailing launch per panel (depth 1).
    int last_ev = -1;  // last panel with a recorded ev_tu (U(p,p+2) at depth 2, the whole trailing update at depth 1)
    for (int p = 0; p < NP; p++) {
        const int p0 = p * PB;
        const int pend = (p0 + PB < T) ? p0 + PB : T;
        GPP_TRY(panel_factor(A, M, ld, T, p0, pend, logdet_part, info, la.side, oz));
        // with U(p,p+1) on the INT8-sliced GEMM the digit planes of the whole panel (rows pend..T) are cut here, on the
        // side stream, and the main stream's updates reuse them
        const bool ozp = oz && oz->next_on_oz && oz_use_trailing(oz, T, pend);
        if (ozp) GPP_TRY(oz_split_panel(*oz, A, ld, T, p0, pend, pend, p & 3, la.side));
        GPP_TRY(cudaEventRecord(la.ev_pf[p], la.side));
        if (pend >= T) break;
        if (overlap && !la.inv_pending && pend >= H) {
            // the first H tile columns of L are final: their share of L^-1 runs behind the rest of the factorisation
            GPP_TRY(cudaStreamWaitEvent(la.inv, la.ev_pf[p], 0));
            GPP_TRY(trtri_early(A, M, X, ld, T, la.inv, oz));
            GPP_TRY(cudaEventRecord(la.inv_done, la.inv));
            la.inv_pending = true;
        }
        const int nend = (pend + PB < T) ? pend + PB : T;
        if (last_ev >= 0) GPP_TRY(cudaStreamWaitEvent(la.side, la.ev_tu[last_ev], 0));
        if (ozp) GPP_TRY(oz_trailing_update(*oz, A, ld, T, p0, pend, pend, nend, p & 3, la.side));  // U(p,p+1)
        else GPP_TRY(trailing_update(A, ld, T, p0, pend, pend, nend, la.side));
        if (nend < T) {
            GPP_TRY(cudaStreamWaitEvent(st, la.ev_pf[p], 0));
            if (oz_use_trailing(oz, T, nend)) {
                // the bulk of the trailing update on the INT8-sliced GEMM: digit planes of the panel rows nend..T once,
                // then U(p,p+2) and U(p,p+3..) as integer GEMMs
                if (!ozp) GPP_TRY(oz_split_panel(*oz, A, ld, T, p0, pend, nend, p & 3, st));
                const int n2end = (deep && nend + PB < T) ? nend + PB : T;
                GPP_TRY(oz_trailing_update(*oz, A, ld, T, p0, pend, nend, n2end, p & 3, st));
                GPP_TRY(cudaEventRecord(la.ev_tu[p], st));
                if (n2end < T) GPP_TRY(oz_trailing_update(*oz, A, ld, T, p0, pend, n2end, T, p & 3, st));
            } else if (deep) {
                const int n2end = (nend + PB < T) ? nend + PB : T;
                GPP_TRY(trailing_update(A, ld, T, p0, pend, nend, n2end, st));  // U(p,p+2)
                GPP_TRY(cudaEventRecord(la.ev_tu[p], st));
                GPP_TRY(trailing_update(A, ld, T, p0, pend, n2end, T, st));  // U(p,p+3..)
            } else {
                GPP_TRY(trailing_update(A, ld, T, p0, pend, nend, T, st));
                GPP_TRY(cudaEventRecord(la.ev_tu[p], st));
            }
            last_ev = p;
        }
    }
    GPP_TRY(cudaEventRecord(la.join, la.side));
    GPP_TRY(cudaStreamWaitEvent(st, la.join, 0));
    return cudaSuccess;
}

// defined below
inline cudaError_t trtri_doubling(const double* L, double* M, double* X, int ld, int T, cudaStream_t st, OzCtx* oz = nullptr);
// M (diagonal 128-blocks already hold L_kk^-1) <- L^-1 (lower); X is an N x N scratch.
// One level of the recursive doubling on the groups [g_lo, g_hi) of 2*hb tiles each:
//   X21 = L21 * M11 (part & 1), then M21 = -M22 * X21 (part & 2); groups are independent (batched launch).
inline cudaError_t trtri_level(const double* L, double* M, double* X, int ld, int T, int hb, int g_lo, int g_hi,
                               int part, cudaStream_t st, int max_ctas = 0, OzCtx* oz = nullptr) {
    int nb = 0, last_s2 = 0;  // groups of the range with a non-empty second half
    for (int gidx = g_lo; gidx < g_hi; gidx++) {
        int s2 = T - (gidx * 2 * hb + hb);
        if (s2 <= 0) break;
        if (s2 > hb) s2 = hb;
        nb++;
        last_s2 = s2;
    }
    if (nb == 0) return cudaSuccess;
    if (oz_use_level(oz, hb)) return oz_trtri_level(*oz, L, M, X, ld, hb, g_lo, nb, last_s2, part, st);
    const long long zs = (long long)2 * hb * TILE * ld + (long long)2 * hb * TILE;  // next group, diagonal step
    const long long base = (long long)g_lo * zs;
    const long long off21 = base + (long long)hb * TILE * ld;                        // block (hb, 0) of the group
    const long long off22 = base + (long long)hb * TILE * ld + (long long)hb * TILE;
    if (part & 1) {   // X21 = L21 * M11 ; M11 lower: k-blocks [tj, hb)
        GemmOp op = gemm_default();
        op.A = L + off21;
        op.lda = ld;
        op.a_zs = zs;
        op.B = M + base;
        op.ldb = ld;
        op.b_zs = zs;
        op.C = X + off21;
        op.ldc = ld;
        op.c_zs = zs;
        op.tiles_m = hb;
        op.tiles_m_last = last_s2;
        op.tiles_n = hb;
        op.klo_sel = KSEL_TJ;
        op.klo_c = 0;
        op.khi_sel = KSEL_CONST;
        op.khi_c = hb;
        op.max_ctas = (nb == 1) ? max_ctas : 0;
        GPP_TRY(launch_gemm(op, true, false, nb, st));
    }
    if (part & 2) {   // M21 = -M22 * X21 ; M22 lower: k-blocks [0, ti+1)
        GemmOp op = gemm_default();
        op.A = M + off22;
        op.lda = ld;
        op.a_zs = zs;
        op.B = X + off21;
        op.ldb = ld;
        op.b_zs = zs;
        op.C = M + off21;
        op.ldc = ld;
        op.c_zs = zs;
        op.tiles_m = hb;
        op.tiles_m_last = last_s2;
        op.tiles_n = hb;
        op.klo_sel = KSEL_CONST;
        op.klo_c = 0;
        op.khi_sel = KSEL_TI;
        op.khi_c = 1;
        op.alpha = -1.0;
        op.max_ctas = (nb == 1) ? max_ctas : 0;
        GPP_TRY(launch_gemm(op, true, false, nb, st));
    }
    return cudaSuccess;
}

inline cudaError_t trtri_doubling(const double* L, double* M, double* X, int ld, int T, cudaStream_t st,
                                  OzCtx* oz) {
    for (int hb = 1; hb < T; hb *= 2)
        GPP_TRY(trtri_level(L, M, X, ld, T, hb, 0, (T + 2 * hb - 1) / (2 * hb), 3, st, 0, oz));
    return cudaSuccess;
}

// Split of the same computation around H = largest power of two below T, so that the part that only needs the
// first H tile columns of L can run while the factorisation is still working on the rest (where it is
// latency-bound and leaves SMs idle):
//   early (needs L[:, 0:H] final):  L11^-1 for the leading H tiles (all levels hb < H on the groups inside [0,H))
//                                   and X21 = L[H:T, 0:H] * M11 (first half of the top level)
//   late  (needs all of L):         the levels hb < H on the groups inside [H,T), then M21 = -M22 * X21
inline int trtri_split_point(int T) {
    int H = 1;
    while (H * 2 < T) H *= 2;
    return (T >= 2) ? H : 0;
}
inline cudaError_t trtri_early(const double* L, double* M, double* X, int ld, int T, cudaStream_t st, OzCtx* oz = nullptr) {
    const int H = trtri_split_point(T);
    if (H == 0) return cudaSuccess;
    for (int hb = 1; hb < H; hb *= 2)
        GPP_TRY(trtri_level(L, M, X, ld, T, hb, 0, H / (2 * hb), 3, st, 0, oz));
    return trtri_level(L, M, X, ld, T, H, 0, 1, 1, st, 0, oz);
}
inline cudaError_t trtri_late(const double* L, double* M, double* X, int ld, int T, cudaStream_t st, OzCtx* oz = nullptr) {
    const int H = trtri_split_point(T);
    if (H == 0) return cudaSuccess;
    for (int hb = 1; hb < H; hb *= 2)
        GPP_TRY(trtri_level(L, M, X, ld, T, hb, H / (2 * hb), (T + 2 * hb - 1) / (2 * hb), 3, st, 0, oz));
    return trtri_level(L, M, X, ld, T, H, 0, 1, 2, st, 0, oz);
}


// ---------------------------------------------------------------------------------------------
// Lazy-panel variant for the INT8-sliced path.  With the trailing updates ~3x faster than on DMMA, the panel chain of
// potrf_lookahead (leaf / TRSM / in-panel updates over ALL rows below: ~2.3 ms per 1536-column panel) became the
// critical path.  Here the chain only factors the DIAGONAL block of a panel (12 x 12 tiles) and inverts it
// (W = L_pp^-1, recursive doubling inside the block -- these are final entries of L^-1); the rows below are then
// solved in one integer GEMM, L[rows, panel] = A[rows, panel] W^T, which is throughput work:
//
//   side:  B(0) s1(0) u1(0) B(1) [wait m1(0)] s1(1) [wait m2(0)] u1(1) B(2) ...
//   main:       [wait B(0)] s2(0) [wait s1(0)] m1(0) m2(0) m3(0)   [wait B(1)] s2(1) ...
//
//   B(p)   factor + invert the diagonal block of panel p, cut W into digit planes
//   s1(p)  solve the rows of the NEXT diagonal block (tile rows [pend, nend)), cut them into planes
//   u1(p)  update of block (p+1, p+1) with panel p                     -> B(p+1) can start
//   s2(p)  solve the remaining rows [nend, T), cut them into planes
//   m1(p)  update of tile-column block p+1, rows >= nend               -> s1(p+1) can start
//   m2(p)  update of tile-column block p+2, rows >= nend               -> u1(p+1) can start
//   m2b(p) update of tile-column block p+3
//   m3(p)  update of everything to the right of block p+3, issued after the urgent pieces of panel p+1
inline cudaError_t potrf_lazy(double* A, double* M, int ld, int T, double* logdet_part, int* info, cudaStream_t st,
                              CholLookahead& la, double* X, OzCtx& oz) {
    const int PB = oz.lazy_pb;
    const int NP = (T + PB - 1) / PB;
    if (NP > la.panels || PB > OzCtx::LAZY_PB || PB < 2) return cudaErrorInvalidValue;
    const int H = trtri_split_point(T);
    const bool overlap = g_overlap_inverse && X != nullptr && H > 0 && NP > 1;
    la.inv_pending = false;
    GPP_TRY(cudaEventRecord(la.fork, st));
    GPP_TRY(cudaStreamWaitEvent(la.side, la.fork, 0));
    int def_p0 = -1, def_pend = 0, def_c0 = 0, def_slot = 0;   // deferred bulk update
    for (int p = 0; p < NP; p++) {
        const int p0 = p * PB;
        const int pend = (p0 + PB < T) ? p0 + PB : T;
        const int nend = (pend + PB < T) ? pend + PB : T;
        const int n2end = (nend + PB < T) ? nend + PB : T;
        const int buf = p & 1, slot = p & 3;
        // ---- B(p): diagonal block on the chain: one dataflow launch (or the launch-per-step chain with row limit pend) ----
        if (la.blk_ctas > 0 && pend - p0 <= 16)
            GPP_TRY(launch_block_potrf(A, M, ld, p0, pend - p0, logdet_part, info, la.blk_flags, ++la.blk_epoch, la.blk_ctas,
                                       la.side));
        else
            GPP_TRY(panel_factor(A, M, ld, pend, p0, pend, logdet_part, info, la.side, nullptr));
        if (pend < T) {
            const long long o = (long long)p0 * TILE * ld + (long long)p0 * TILE;
            GPP_TRY(trtri_doubling(A + o, M + o, X + o, ld, pend - p0, la.side, nullptr));
            GPP_TRY(oz_split_w(oz, M + o, ld, pend - p0, buf, la.side));
        }
        GPP_TRY(cudaEventRecord(la.ev_pf[p], la.side));
        if (pend >= T) break;
        // ---- side: the pieces the next diagonal block waits for ----
        if (p >= 1) GPP_TRY(cudaStreamWaitEvent(la.side, la.ev_m1[p - 1], 0));
        GPP_TRY(oz_panel_solve(oz, A, ld, p0, pend, pend, nend, buf, 4, la.side));                 // s1
        GPP_TRY(oz_split_panel_rows(oz, A, ld, p0, pend, pend, nend, slot, la.side));
        GPP_TRY(cudaEventRecord(la.ev_s1[p], la.side));
        if (p >= 1) GPP_TRY(cudaStreamWaitEvent(la.side, la.ev_tu[p - 1], 0));
        GPP_TRY(oz_update_region(oz, A, ld, p0, pend, pend, nend, pend, nend, slot, la.side));      // u1
        // ---- main: throughput work; the bulk update m3 of a panel is issued one panel late, behind the next
        // panel's urgent pieces, so that the chain never queues behind it ----
        GPP_TRY(cudaStreamWaitEvent(st, la.ev_pf[p], 0));
        const int n3end = (n2end + PB < T) ? n2end + PB : T;
        if (nend < T) {
            GPP_TRY(oz_panel_solve(oz, A, ld, p0, pend, nend, T, buf, 5, st, true));                // s2
            GPP_TRY(oz_split_panel_rows(oz, A, ld, p0, pend, nend, T, slot, st));
            GPP_TRY(cudaStreamWaitEvent(st, la.ev_s1[p], 0));
            GPP_TRY(oz_update_region(oz, A, ld, p0, pend, nend, T, pend, nend, slot, st, true));    // m1
            GPP_TRY(cudaEventRecord(la.ev_m1[p], st));
            if (overlap && !la.inv_pending && pend >= H) {
                // every row of the first H tile columns of L is final: their share of L^-1 runs behind the rest
                GPP_TRY(cudaStreamWaitEvent(la.inv, la.ev_m1[p], 0));
                GPP_TRY(trtri_early(A, M, X, ld, T, la.inv, &oz));
                GPP_TRY(cudaEventRecord(la.inv_done, la.inv));
                la.inv_pending = true;
            }
            GPP_TRY(oz_update_region(oz, A, ld, p0, pend, nend, T, nend, n2end, slot, st, true));   // m2
            GPP_TRY(cudaEventRecord(la.ev_tu[p], st));
            if (n2end < T) GPP_TRY(oz_update_region(oz, A, ld, p0, pend, n2end, T, n2end, n3end, slot, st, true));  // m2b
        } else {
            GPP_TRY(cudaEventRecord(la.ev_m1[p], st));
            GPP_TRY(cudaEventRecord(la.ev_tu[p], st));
        }
        if (def_p0 >= 0) {   // m3 of the previous panel
            GPP_TRY(oz_update_region(oz, A, ld, def_p0, def_pend, def_c0, T, def_c0, T, def_slot, st, true));
            def_p0 = -1;
        }
        if (n3end < T) {
            def_p0 = p0;
            def_pend = pend;
            def_c0 = n3end;
            def_slot = slot;
        }
    }
    if (def_p0 >= 0) GPP_TRY(oz_update_region(oz, A, ld, def_p0, def_pend, def_c0, T, def_c0, T, def_slot, st, true));
    GPP_TRY(cudaEventRecord(la.join, la.side));
    GPP_TRY(cudaStreamWaitEvent(st, la.join, 0));
    return cudaSuccess;
}

// Kinv = M^T M over the lower tiles; M lower: k-blocks [ti, T).  The hot path reads lower tiles only (the gradient
// pass and the noise-gradient diagonal), so the upper triangle is not written unless `mirror` is set: the mirrored
// store was 3.6x the algorithmic DRAM traffic of this launch (strided 8-byte stores, profiles/dgemm_traffic.json).
inline cudaError_t lauum_full(const double* M, double* Kinv, int ld, int T, cudaStream_t st, int mirror = 0,
                              OzCtx* oz = nullptr) {
    if (!mirror && oz_use_lauum(oz, T)) return oz_lauum(*oz, M, Kinv, ld, T, st);
    GemmOp op = gemm_default();
    op.A = M;
    op.lda = ld;
    op.B = M;
    op.ldb = ld;
    op.C = Kinv;
    op.ldc = ld;
    op.map = MAP_TRI;
    op.tiles_m = op.tiles_m_last = T;
    op.tiles_n = T;
    op.klo_sel = KSEL_TI;
    op.klo_c = 0;
    op.khi_sel = KSEL_CONST;
    op.khi_c = T;
    op.mirror = mirror;
    return launch_gemm(op, false, false, 1, st);
}

}  // namespace gpp
