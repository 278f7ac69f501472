// The three O(N^3) stages on the INT8-sliced tcgen05 GEMM (oz_gemm.cuh): trailing updates of the factorisation,
// the levels of the recursive-doubling triangular inverse and K^-1 = M^T M.  chol.cuh calls these instead of the
// DMMA launches when a handle carries an OzCtx and the shape is large enough to fill the machine.
//
// Digit planes live in three N x N x 7 int8 buffers, addressed with the coordinates of the matrix they are cut from:
//   PP  panel planes     (row, k) of L          -- trailing updates  A[i,j] -= sum_k L[i,k] L[j,k], k in the panel
//   PA  A-operand planes (row, k) of L / M      -- inverse levels: L21, M22
//   PB  B-operand planes (col, k) of M / X      -- inverse levels: M11^T, X21^T; K^-1: M^T
// The factorisation (main stream) and the early part of the inverse (low-priority stream) run concurrently, hence
// separate buffers; the panel scales rotate over four arrays because up to three panels are in flight with the
// depth-2 look-ahead.
#pragma once
#include "oz_split.cuh"

namespace gpp {

// Which work of the three stages runs on the INT8-sliced GEMM, and how (int fields only: gpp_create compares
// configurations with memcmp).  The member initialisers are the production configuration.
struct OzSchedule {
    int min_trailing_tiles = 12;   // smaller trailing matrices stay on DMMA (too few 128x64 items for 148 SMs)
                                   // (GPP_OZ_MIN_TRAIL)
    int min_level_tiles = 4;       // inverse levels below this half-width stay on DMMA (K < 512) (GPP_OZ_MIN_LEVEL)
    int next_on_oz = 1;            // U(p,p+1), the update of the next panel's own columns, also runs here (GPP_OZ_NEXT)
    int inner_min_k = 4;           // in-panel (recursive) updates with K >= this many tiles run here; 0 = never
                                   // (GPP_OZ_INNER)
    int kinv_levels = 7;           // significance levels of K^-1 = M^T M (GPP_OZ_KINV_LEVELS).  Its only consumer is the
                                   // gradient trace (tolerance 1e-8 of the gradient's max-norm): with 6 levels (21 of 28
                                   // plane pairs) the product takes 11.1 instead of 13.4 ms at N = 16384 and the gradient
                                   // moves by 6.6e-11 instead of 2.9e-13.  Default 7: both arithmetics then agree at the
                                   // FP64 rounding level and multi-start fits follow the same L-BFGS-B paths
    int lazy_min_tiles = 96;       // lazy panels (potrf_lazy) from N = 12288 (GPP_OZ_LAZY_MIN); below, 512-column panels
                                   // of the look-ahead schedule keep the chain shorter (measured: N = 8192 12.7 vs 14.0 ms,
                                   // N = 12288 28.5 vs 27.9, N = 16384 55.3 vs 54.4)
    int lazy_pb = 12;              // lazy panel width in 128-tiles, 2 .. OzCtx::LAZY_PB (GPP_OZ_LAZY_PB)
    int stagger = 6000;            // ns per 128-block of K: estimated duration of one 128x128 item, see OzGemmOp.stagger_ns
                                   // (GPP_OZ_STAGGER)
};

struct OzCtx {
    bool ready = false;
    int np = 0, T = 0;
    OzPlanes PP, PA, PB;
    // [0..3]: factored panels by panel index mod 4; [4]: side-stream scratch (in-panel updates, panel rows before their
    // solve); [5]: main-stream scratch (panel rows before their solve)
    double* pscale[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    // lazy panels: only the diagonal block of a panel is factored on the latency-bound chain; the rows below are solved
    // against its explicit inverse W = L_pp^-1 by one integer GEMM.  W's digit planes, double-buffered by panel parity:
    static constexpr int LAZY_PB = 16;     // widest panel in 128-tiles (sizes the W planes)
    OzPlanes PW[2];
    CUtensorMap mPW_b[2];
    CUtensorMap mPP_a, mPP_b, mPA_a, mPB_a, mPB_b;
    OzSchedule sched;
    size_t bytes = 0;

    static cudaError_t alloc_planes(OzPlanes& P, long long np, size_t& bytes) {
        P.rows = np;
        P.pitch = np;
        cudaError_t e = cudaMalloc(&P.planes, (size_t)OZ_S * np * np);
        if (e != cudaSuccess) return e;
        // never-written regions (strict upper tiles) may be touched by TMA boxes only through K ranges that the
        // callers exclude; zero them once anyway so that nothing undefined can enter an integer accumulator
        e = cudaMemset(P.planes, 0, (size_t)OZ_S * np * np);
        if (e != cudaSuccess) return e;
        e = cudaMalloc(&P.scale, sizeof(double) * np);
        if (e != cudaSuccess) return e;
        e = cudaMalloc(&P.colmax, sizeof(unsigned long long) * np);
        bytes += (size_t)OZ_S * np * np + 16 * (size_t)np;
        return e;
    }
    static void free_planes(OzPlanes& P) {
        if (P.planes) cudaFree(P.planes);
        if (P.scale) cudaFree(P.scale);
        if (P.colmax) cudaFree(P.colmax);
        P = OzPlanes();
    }

    cudaError_t init(int np_) {
        np = np_;
        T = np / TILE;
        cudaError_t e;
        if ((e = alloc_planes(PP, np, bytes)) != cudaSuccess) return e;
        if ((e = alloc_planes(PA, np, bytes)) != cudaSuccess) return e;
        if ((e = alloc_planes(PB, np, bytes)) != cudaSuccess) return e;
        for (int i = 0; i < 6; i++)
            if ((e = cudaMalloc(&pscale[i], sizeof(double) * np)) != cudaSuccess) return e;
        for (int i = 0; i < 2; i++) {
            const long long wr = (long long)LAZY_PB * TILE;
            if ((e = alloc_planes(PW[i], wr, bytes)) != cudaSuccess) return e;
            if ((e = oz_make_map(&mPW_b[i], PW[i].planes, wr, (long long)OZ_S * wr, wr, OZ_BN)) != cudaSuccess) return e;
        }
        const long long rows = (long long)OZ_S * np;
        if ((e = oz_make_map(&mPP_a, PP.planes, np, rows, np, OZ_BM)) != cudaSuccess) return e;
        if ((e = oz_make_map(&mPP_b, PP.planes, np, rows, np, OZ_BN)) != cudaSuccess) return e;
        if ((e = oz_make_map(&mPA_a, PA.planes, np, rows, np, OZ_BM)) != cudaSuccess) return e;
        if ((e = oz_make_map(&mPB_a, PB.planes, np, rows, np, OZ_BM)) != cudaSuccess) return e;
        if ((e = oz_make_map(&mPB_b, PB.planes, np, rows, np, OZ_BN)) != cudaSuccess) return e;
        ready = true;
        return cudaSuccess;
    }
    void destroy() {
        free_planes(PP);
        free_planes(PA);
        free_planes(PB);
        for (int i = 0; i < 6; i++) {
            if (pscale[i]) cudaFree(pscale[i]);
            pscale[i] = nullptr;
        }
        free_planes(PW[0]);
        free_planes(PW[1]);
        ready = false;
    }
};

// digit planes of the factored panel p (tile columns [p0, pend), tile rows r0..T) -- the operand of every
// trailing update with that panel on the main stream
inline cudaError_t oz_split_panel(OzCtx& oz, const double* A, int ld, int T, int p0, int pend, int r0, int slot,
                                  cudaStream_t st) {
    if (r0 >= T) return cudaSuccess;
    OzPlanes pp = oz.PP;
    pp.scale = oz.pscale[slot];   // indexed by absolute plane row like PP.scale
    const int rows = (T - r0) * TILE;
    return oz_split_rows(A + (long long)r0 * TILE * ld + (long long)p0 * TILE, ld, 0, rows, rows, (pend - p0) * TILE, pp,
                         (long long)r0 * TILE, (long long)p0 * TILE, 0, 0, 1, st);
}

inline bool oz_use_trailing(const OzCtx* oz, int T, int c0) { return oz && oz->ready && (T - c0) >= oz->sched.min_trailing_tiles; }

// C[i,j] -= sum_{k in [p0,pend)} L[i,k] L[j,k] for tile rows i >= c0, tile columns j in [c0, c1), i >= j
inline cudaError_t oz_trailing_update(OzCtx& oz, double* A, int ld, int T, int p0, int pend, int c0, int c1, int slot,
                                      cudaStream_t st) {
    if (c1 <= c0 || c0 >= T) return cudaSuccess;
    OzGemmOp op = oz_default();
    op.a_plane_rows = op.b_plane_rows = oz.np;
    op.a_row0 = op.b_row0 = c0 * TILE;
    op.a_k0 = op.b_k0 = p0 * TILE;
    op.a_scale = op.b_scale = oz.pscale[slot];
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
    op.stagger_ns = oz.sched.stagger * (pend - p0);
    return launch_oz_gemm(oz.mPP_a, oz.mPP_b, op, 1, st);
}

// general form: C[i,j] -= sum_{k in [p0,pend)} L[i,k] L[j,k] for tile rows i in [r0, r1), tile columns j in [c0, c1), i >= j
// (r0 >= c0; digit planes and scales of panel slot `slot` must cover rows [c0, c1) and [r0, r1))
inline cudaError_t oz_update_region(OzCtx& oz, double* A, int ld, int p0, int pend, int r0, int r1, int c0, int c1, int slot,
                                    cudaStream_t st, bool stagger = false) {
    if (c1 <= c0 || r1 <= r0) return cudaSuccess;
    OzGemmOp op = oz_default();
    op.a_plane_rows = op.b_plane_rows = oz.np;
    op.a_row0 = r0 * TILE;
    op.b_row0 = c0 * TILE;
    op.a_k0 = op.b_k0 = p0 * TILE;
    op.a_scale = op.b_scale = oz.pscale[slot];
    op.C = A + (long long)r0 * TILE * ld + (long long)c0 * TILE;
    op.ldc = ld;
    op.tiles_m = op.tiles_m_last = r1 - r0;
    op.tiles_n = c1 - c0;
    op.klo_c = 0;
    op.khi_c = pend - p0;
    op.alpha = -1.0;
    op.beta = 1.0;
    if (r0 == c0 && r1 - r0 == c1 - c0) {
        op.map = MAP_TRI;
    } else {
        op.lower_filter = 1;
        op.lower_off = r0 - c0;
    }
    if (stagger) op.stagger_ns = oz.sched.stagger * (pend - p0);
    return launch_oz_gemm(oz.mPP_a, oz.mPP_b, op, 1, st);
}

// digit planes of W = L_pp^-1 (lower triangular pw x pw tiles, given in M's diagonal block) into PW[buf]
inline cudaError_t oz_split_w(OzCtx& oz, const double* Wblk, int ld, int pw, int buf, cudaStream_t st) {
    return oz_split_rows(Wblk, ld, 0, pw * TILE, pw * TILE, pw * TILE, oz.PW[buf], 0, 0, 0, 0, 1, st);
}

// panel rows [r0, r1) x tile columns [p0, pend):  X = A W^T in place (X[i,c] = sum_{k <= c} A[i,k] W[c,k]); the rows are
// cut into digit planes first (scratch scale slot `pre_slot`), so writing the result over A is safe
inline cudaError_t oz_panel_solve(OzCtx& oz, double* A, int ld, int p0, int pend, int r0, int r1, int buf, int pre_slot,
                                  cudaStream_t st, bool stagger = false) {
    if (r1 <= r0) return cudaSuccess;
    OzPlanes pp = oz.PP;
    pp.scale = oz.pscale[pre_slot];
    const int rows = (r1 - r0) * TILE;
    cudaError_t e = oz_split_rows(A + (long long)r0 * TILE * ld + (long long)p0 * TILE, ld, 0, rows, rows, (pend - p0) * TILE,
                                  pp, (long long)r0 * TILE, (long long)p0 * TILE, 0, 0, 1, st);
    if (e != cudaSuccess) return e;
    OzGemmOp op = oz_default();
    op.a_plane_rows = oz.np;
    op.b_plane_rows = OzCtx::LAZY_PB * TILE;
    op.a_row0 = r0 * TILE;
    op.a_k0 = p0 * TILE;
    op.b_row0 = 0;
    op.b_k0 = 0;
    op.a_scale = oz.pscale[pre_slot];
    op.b_scale = oz.PW[buf].scale;
    op.C = A + (long long)r0 * TILE * ld + (long long)p0 * TILE;
    op.ldc = ld;
    op.tiles_m = op.tiles_m_last = r1 - r0;
    op.tiles_n = pend - p0;
    op.klo_sel = KSEL_CONST;
    op.klo_c = 0;
    op.khi_sel = KSEL_TJ;
    op.khi_c = 1;
    if (stagger) op.stagger_ns = oz.sched.stagger * (pend - p0) / 2;
    return launch_oz_gemm(oz.mPP_a, oz.mPW_b[buf], op, 1, st);
}

// digit planes of solved panel rows [r0, r1) (operand of the trailing updates), scale slot `slot`
inline cudaError_t oz_split_panel_rows(OzCtx& oz, const double* A, int ld, int p0, int pend, int r0, int r1, int slot,
                                       cudaStream_t st) {
    if (r1 <= r0) return cudaSuccess;
    OzPlanes pp = oz.PP;
    pp.scale = oz.pscale[slot];
    const int rows = (r1 - r0) * TILE;
    return oz_split_rows(A + (long long)r0 * TILE * ld + (long long)p0 * TILE, ld, 0, rows, rows, (pend - p0) * TILE, pp,
                         (long long)r0 * TILE, (long long)p0 * TILE, 0, 0, 1, st);
}

inline bool oz_use_level(const OzCtx* oz, int hb) { return oz && oz->ready && hb >= oz->sched.min_level_tiles && hb <= 128; }

// one level of the recursive doubling (see trtri_level in chol.cuh): X21 = L21 * M11 (part & 1), M21 = -M22 * X21 (part & 2)
inline cudaError_t oz_trtri_level(OzCtx& oz, const double* L, double* M, double* X, int ld, int hb, int g_lo, int nb,
                                  int last_s2, int part, cudaStream_t st) {
    const long long zs = (long long)2 * hb * TILE * ld + (long long)2 * hb * TILE;
    const long long base = (long long)g_lo * zs;
    const long long off21 = base + (long long)hb * TILE * ld;
    const long long off22 = off21 + (long long)hb * TILE;
    const int g0 = g_lo * 2 * hb * TILE;     // first row / column of the first group
    const int h = hb * TILE, step = 2 * hb * TILE;
    cudaError_t e;
    if (part & 1) {
        // A = L21 (rows g0+h.., k = columns g0..g0+h), B = M11^T (rows = columns of M11, k = rows of M11, k >= row)
        if ((e = oz_split_rows(L + off21, ld, zs, h, last_s2 * TILE, h, oz.PA, g0 + h, g0, step, step, nb, st)) != cudaSuccess)
            return e;
        if ((e = oz_split_cols(M + base, ld, zs, h, h, h, 1, oz.PB, g0, g0, step, step, nb, st)) != cudaSuccess) return e;
        OzGemmOp op = oz_default();
        op.a_plane_rows = op.b_plane_rows = oz.np;
        op.a_row0 = g0 + h;
        op.a_k0 = g0;
        op.b_row0 = g0;
        op.b_k0 = g0;
        op.a_zs_row = op.a_zs_k = op.b_zs_row = op.b_zs_k = step;
        op.a_scale = oz.PA.scale;
        op.b_scale = oz.PB.scale;
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
        if ((e = launch_oz_gemm(oz.mPA_a, oz.mPB_b, op, nb, st)) != cudaSuccess) return e;
    }
    if (part & 2) {
        // A = M22 (rows g0+h.., k = columns g0+h.. up to the row), B = X21^T (rows = columns g0.. of X21, k = rows g0+h..)
        if ((e = oz_split_rows(M + off22, ld, zs, h, last_s2 * TILE, h, oz.PA, g0 + h, g0 + h, step, step, nb, st,
                               last_s2 * TILE)) != cudaSuccess)
            return e;
        if ((e = oz_split_cols(X + off21, ld, zs, h, last_s2 * TILE, h, 0, oz.PB, g0, g0 + h, step, step, nb, st)) != cudaSuccess)
            return e;
        OzGemmOp op = oz_default();
        op.a_plane_rows = op.b_plane_rows = oz.np;
        op.a_row0 = g0 + h;
        op.a_k0 = g0 + h;
        op.b_row0 = g0;
        op.b_k0 = g0 + h;
        op.a_zs_row = op.a_zs_k = op.b_zs_row = op.b_zs_k = step;
        op.a_scale = oz.PA.scale;
        op.b_scale = oz.PB.scale;
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
        if ((e = launch_oz_gemm(oz.mPA_a, oz.mPB_b, op, nb, st)) != cudaSuccess) return e;
    }
    return cudaSuccess;
}

inline bool oz_use_lauum(const OzCtx* oz, int T) { return oz && oz->ready && T >= 24; }

// Kinv (lower tiles) = M^T M, M lower triangular
inline cudaError_t oz_lauum(OzCtx& oz, const double* M, double* Kinv, int ld, int T, cudaStream_t st) {
    cudaError_t e = oz_split_cols(M, ld, 0, T * TILE, T * TILE, T * TILE, 1, oz.PB, 0, 0, 0, 0, 1, st);
    if (e != cudaSuccess) return e;
    OzGemmOp op = oz_default();
    op.a_plane_rows = op.b_plane_rows = oz.np;
    op.a_scale = op.b_scale = oz.PB.scale;
    op.C = Kinv;
    op.ldc = ld;
    op.map = MAP_TRI;
    op.tiles_m = op.tiles_m_last = T;
    op.tiles_n = T;
    op.klo_sel = KSEL_TI;
    op.klo_c = 0;
    op.khi_sel = KSEL_CONST;
    op.khi_c = T;
    op.levels = oz.sched.kinv_levels;
    // K ranges longer than 128 blocks (N > 16384) are accumulated in segments: |digit| <= 128, so 16384 products per
    // int32 accumulation cannot overflow
    for (int k0 = 0; k0 < T; k0 += 128) {
        op.k_min = k0;
        op.k_max = (k0 + 128 < T) ? k0 + 128 : T;
        op.beta = (k0 == 0) ? 0.0 : 1.0;
        if ((e = launch_oz_gemm(oz.mPB_a, oz.mPB_b, op, 1, st)) != cudaSuccess) return e;
    }
    return cudaSuccess;
}

}  // namespace gpp
