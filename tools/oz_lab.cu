// Development bench for the INT8-sliced FP64 GEMM (oz_gemm.cuh / oz_split.cuh); not part of the product library.
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -lineinfo -o tools/oz_lab tools/oz_lab.cu
//   ./tools/oz_lab [check|ragged|maps|segments|limits|exponents|perf|all]
// check: digit planes against a host re-computation, the integer GEMM against an exact host sum over the planes,
//        the scaled result against a long-double product, transposed split against the row split, the
//        lower-triangular K-range map (K^-1 = M^T M shape) and the batched form.
// The check groups below print one line per check (observed error, its bound) and "<group>: ok" or "<group>: FAILED":
//   ragged     the batched inverse levels of oz_trtri_level with a short last group (tiles_m_last = 1 and hb - 1)
//   maps       oz_update_region with lower_off > 0 (filtered tiles untouched), oz_panel_solve (KSEL_TJ upper bound,
//              B planes of LAZY_PB * 128 rows)
//   segments   a K range of 2 * 128 + 10 blocks accumulated in k_min / k_max segments, items with empty ranges
//   limits     digit planes written directly: the largest int32 accumulation (K = 16384, every pair product
//              positive) in closed form, random digits against int64 host sums at 7, 6 and 5 levels
//   exponents  split_rows / split_cols of rows with maxima from 2^-1074 to 2^996, NaN / Inf / zero rows, and the
//              product of such rows
// perf:  timings of square / SYRK / LAUUM shapes against the DMMA kernel.
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "../gp-plus_b200/csrc/oz_chol.cuh"

using namespace gpp;

#define CHECK(x)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (x);                                                                      \
        if (e_ != cudaSuccess) {                                                                   \
            fprintf(stderr, "%s:%d %s -> %s\n", __FILE__, __LINE__, #x, cudaGetErrorString(e_)); \
            exit(1);                                                                               \
        }                                                                                          \
    } while (0)

static double urand(unsigned long long& s) {
    s = s * 6364136223846793005ull + 1442695040888963407ull;
    return ((double)(s >> 11) / 9007199254740992.0) * 2.0 - 1.0;
}

static OzPlanes alloc_planes(long long rows, long long pitch) {
    OzPlanes P;
    P.rows = rows;
    P.pitch = pitch;
    CHECK(cudaMalloc(&P.planes, (size_t)OZ_S * rows * pitch));
    CHECK(cudaMemset(P.planes, 0, (size_t)OZ_S * rows * pitch));
    CHECK(cudaMalloc(&P.scale, sizeof(double) * rows));
    CHECK(cudaMemset(P.scale, 0, sizeof(double) * rows));
    CHECK(cudaMalloc(&P.colmax, sizeof(unsigned long long) * rows));
    return P;
}
static void free_planes(OzPlanes& P) {
    cudaFree(P.planes);
    cudaFree(P.scale);
    cudaFree(P.colmax);
}

// host digits of one value
static void host_digits(double x, double scale, int8_t* d) {
    long long v = (long long)floor(ldexp(x / scale, 56));
    for (int p = OZ_S - 1; p >= 0; p--) {
        long long lo = (long long)(int8_t)(v & 0xff);
        d[p] = (int8_t)lo;
        v = (v - lo) >> 8;
    }
}

static int check_small() {
    int fails = 0;
    const int M = 256, N = 256, K = 256;
    std::vector<double> A((size_t)M * K), B((size_t)N * K), At((size_t)K * M);
    unsigned long long seed = 12345;
    for (int r = 0; r < M; r++) {
        const double rs = pow(10.0, 3.0 * urand(seed));
        for (int k = 0; k < K; k++) A[(size_t)r * K + k] = rs * urand(seed) * ((k % 7 == 0) ? 1e-6 : 1.0);
    }
    for (int r = 0; r < N; r++) {
        const double rs = pow(10.0, 3.0 * urand(seed));
        for (int k = 0; k < K; k++) B[(size_t)r * K + k] = rs * urand(seed);
    }
    for (int r = 0; r < M; r++)
        for (int k = 0; k < K; k++) At[(size_t)k * M + r] = A[(size_t)r * K + k];
    double *dA, *dB, *dAt, *dC;
    CHECK(cudaMalloc(&dA, sizeof(double) * M * K));
    CHECK(cudaMalloc(&dB, sizeof(double) * N * K));
    CHECK(cudaMalloc(&dAt, sizeof(double) * M * K));
    CHECK(cudaMalloc(&dC, sizeof(double) * M * N));
    CHECK(cudaMemcpy(dA, A.data(), sizeof(double) * M * K, cudaMemcpyHostToDevice));
    CHECK(cudaMemcpy(dB, B.data(), sizeof(double) * N * K, cudaMemcpyHostToDevice));
    CHECK(cudaMemcpy(dAt, At.data(), sizeof(double) * M * K, cudaMemcpyHostToDevice));
    OzPlanes PA = alloc_planes(M, K), PB = alloc_planes(N, K), PAt = alloc_planes(M, K);
    CHECK(oz_split_rows(dA, K, 0, M, M, K, PA, 0, 0, 0, 0, 1, 0));
    CHECK(oz_split_rows(dB, K, 0, N, N, K, PB, 0, 0, 0, 0, 1, 0));
    CHECK(oz_split_cols(dAt, M, 0, K, K, M, 0, PAt, 0, 0, 0, 0, 1, 0));
    CHECK(cudaDeviceSynchronize());
    std::vector<int8_t> hA((size_t)OZ_S * M * K), hB((size_t)OZ_S * N * K), hAt((size_t)OZ_S * M * K);
    std::vector<double> sA(M), sB(N), sAt(M);
    CHECK(cudaMemcpy(hA.data(), PA.planes, hA.size(), cudaMemcpyDeviceToHost));
    CHECK(cudaMemcpy(hB.data(), PB.planes, hB.size(), cudaMemcpyDeviceToHost));
    CHECK(cudaMemcpy(hAt.data(), PAt.planes, hAt.size(), cudaMemcpyDeviceToHost));
    CHECK(cudaMemcpy(sA.data(), PA.scale, sizeof(double) * M, cudaMemcpyDeviceToHost));
    CHECK(cudaMemcpy(sB.data(), PB.scale, sizeof(double) * N, cudaMemcpyDeviceToHost));
    CHECK(cudaMemcpy(sAt.data(), PAt.scale, sizeof(double) * M, cudaMemcpyDeviceToHost));
    // (1) planes against the host digits
    long long bad_digits = 0, bad_t = 0;
    double worst_rep = 0.0;
    for (int r = 0; r < M; r++) {
        double amax = 0.0;
        for (int k = 0; k < K; k++) amax = fmax(amax, fabs(A[(size_t)r * K + k]));
        int ex;
        frexp(amax, &ex);
        const double sc = ldexp(1.0, ex + 2);
        if (sc != sA[r]) bad_digits++;
        if (sAt[r] != sA[r]) bad_t++;
        for (int k = 0; k < K; k++) {
            int8_t d[OZ_S];
            host_digits(A[(size_t)r * K + k], sc, d);
            long double rep = 0.0L;
            for (int p = 0; p < OZ_S; p++) {
                const int8_t g = hA[((size_t)p * M + r) * K + k];
                if (g != d[p]) bad_digits++;
                if (hAt[((size_t)p * M + r) * K + k] != g) bad_t++;
                rep += (long double)g * powl(256.0L, -(p + 1));
            }
            worst_rep = fmax(worst_rep, (double)fabsl(rep * sc - A[(size_t)r * K + k]) / sc);
        }
    }
    printf("split_rows: digit mismatches %lld, representation error / scale %.3e (bound 2^-56 = %.3e)\n", bad_digits,
           worst_rep, ldexp(1.0, -56));
    printf("split_cols: mismatches against split_rows %lld\n", bad_t);
    if (bad_digits || bad_t || worst_rep > ldexp(1.0, -56)) fails++;
    fflush(stdout);

    // (2) GEMM
    CUtensorMap tmA, tmB;
    CHECK(oz_make_map(&tmA, PA.planes, K, (long long)OZ_S * M, K, OZ_BM));
    CHECK(oz_make_map(&tmB, PB.planes, K, (long long)OZ_S * N, K, OZ_BN));
    CHECK(oz_set_attributes());
    OzGemmOp op = oz_default();
    op.a_plane_rows = M;
    op.b_plane_rows = N;
    op.a_scale = PA.scale;
    op.b_scale = PB.scale;
    op.C = dC;
    op.ldc = N;
    op.tiles_m = op.tiles_m_last = M / TILE;
    op.tiles_n = N / TILE;
    op.klo_c = 0;
    op.khi_c = K / TILE;
    CHECK(cudaMemset(dC, 0xff, sizeof(double) * M * N));
    CHECK(launch_oz_gemm(tmA, tmB, op, 1, 0));
    CHECK(cudaDeviceSynchronize());
    printf("oz_gemm small launch done\n");
    fflush(stdout);
    std::vector<double> C((size_t)M * N);
    CHECK(cudaMemcpy(C.data(), dC, sizeof(double) * M * N, cudaMemcpyDeviceToHost));
    double worst_int = 0.0, worst_true = 0.0;
    for (int r = 0; r < M; r++)
        for (int c = 0; c < N; c++) {
            long double lv[OZ_S];
            for (int l = 0; l < OZ_S; l++) lv[l] = 0.0L;
            long double tru = 0.0L, mag = 0.0L;
            for (int k = 0; k < K; k++) {
                tru += (long double)A[(size_t)r * K + k] * (long double)B[(size_t)c * K + k];
                mag += fabsl((long double)A[(size_t)r * K + k] * (long double)B[(size_t)c * K + k]);
            }
            for (int i = 0; i < OZ_S; i++)
                for (int j = 0; i + j < OZ_S; j++) {
                    long long acc = 0;
                    const int8_t* pa = &hA[((size_t)i * M + r) * K];
                    const int8_t* pb = &hB[((size_t)j * N + c) * K];
                    for (int k = 0; k < K; k++) acc += (long long)pa[k] * (long long)pb[k];
                    lv[i + j] += (long double)acc;
                }
            long double s = 0.0L;
            for (int l = OZ_S - 1; l >= 0; l--) s = s / 256.0L + lv[l];
            s = s / 65536.0L * (long double)sA[r] * (long double)sB[c];
            const double got = C[(size_t)r * N + c];
            worst_int = fmax(worst_int, (double)(fabsl(got - s) / (mag + 1e-300L)));
            worst_true = fmax(worst_true, (double)(fabsl(got - tru) / (mag + 1e-300L)));
        }
    printf("oz_gemm 256x256x256 (both / sum|a||b|): vs exact plane sum %.3e; vs long-double product %.3e\n",
           worst_int, worst_true);
    if (!(worst_int < 1e-15) || !(worst_true < 1e-15)) fails++;
    fflush(stdout);

    // (3) alpha / beta and a K sub-range
    {
        std::vector<double> C0((size_t)M * N);
        for (auto& v : C0) v = urand(seed);
        CHECK(cudaMemcpy(dC, C0.data(), sizeof(double) * M * N, cudaMemcpyHostToDevice));
        OzGemmOp o2 = op;
        o2.alpha = -1.0;
        o2.beta = 1.0;
        o2.klo_c = 1;
        o2.khi_c = 2;
        CHECK(launch_oz_gemm(tmA, tmB, o2, 1, 0));
        CHECK(cudaDeviceSynchronize());
        CHECK(cudaMemcpy(C.data(), dC, sizeof(double) * M * N, cudaMemcpyDeviceToHost));
        double worst = 0.0;
        for (int r = 0; r < M; r++)
            for (int c = 0; c < N; c++) {
                long double tru = C0[(size_t)r * N + c], mag = fabs(C0[(size_t)r * N + c]);
                for (int k = 128; k < 256; k++) {
                    tru -= (long double)A[(size_t)r * K + k] * (long double)B[(size_t)c * K + k];
                    mag += fabsl((long double)A[(size_t)r * K + k] * (long double)B[(size_t)c * K + k]);
                }
                worst = fmax(worst, (double)(fabsl(C[(size_t)r * N + c] - tru) / mag));
            }
        printf("alpha=-1 beta=1 K block [1,2): rel %.3e\n", worst);
        if (!(worst < 1e-13)) fails++;
        fflush(stdout);
    }
    cudaFree(dA); cudaFree(dB); cudaFree(dAt); cudaFree(dC);
    free_planes(PA); free_planes(PB); free_planes(PAt);
    return fails;
}

// K^-1 = M^T M shape: M lower triangular (zeros above the diagonal), transposed planes, lower tiles, K range [ti, T)
static int check_lauum(int n) {
    int fails = 0;
    const int T = n / TILE;
    std::vector<double> Mh((size_t)n * n, 0.0);
    unsigned long long seed = 777;
    for (int i = 0; i < n; i++)
        for (int j = 0; j <= i; j++) Mh[(size_t)i * n + j] = urand(seed) * exp(-0.01 * (i - j)) * (i == j ? 3.0 : 1.0);
    double *dM, *dC, *dR;
    CHECK(cudaMalloc(&dM, sizeof(double) * n * n));
    CHECK(cudaMalloc(&dC, sizeof(double) * n * n));
    CHECK(cudaMalloc(&dR, sizeof(double) * n * n));
    CHECK(cudaMemcpy(dM, Mh.data(), sizeof(double) * n * n, cudaMemcpyHostToDevice));
    CHECK(cudaMemset(dC, 0, sizeof(double) * n * n));
    CHECK(cudaMemset(dR, 0, sizeof(double) * n * n));
    OzPlanes P = alloc_planes(n, n);
    CHECK(oz_split_cols(dM, n, 0, n, n, n, 1, P, 0, 0, 0, 0, 1, 0));
    CUtensorMap tmA, tmB;
    CHECK(oz_make_map(&tmA, P.planes, n, (long long)OZ_S * n, n, OZ_BM));
    CHECK(oz_make_map(&tmB, P.planes, n, (long long)OZ_S * n, n, OZ_BN));
    OzGemmOp op = oz_default();
    op.a_plane_rows = op.b_plane_rows = n;
    op.a_scale = op.b_scale = P.scale;
    op.C = dC;
    op.ldc = n;
    op.map = MAP_TRI;
    op.tiles_m = op.tiles_m_last = T;
    op.tiles_n = T;
    op.klo_sel = KSEL_TI;
    op.klo_c = 0;
    op.khi_sel = KSEL_CONST;
    op.khi_c = T;
    CHECK(launch_oz_gemm(tmA, tmB, op, 1, 0));
    // DMMA reference (chol.cuh's lauum shape)
    CHECK(gemm_set_attributes());
    GemmOp g = gemm_default();
    g.A = dM; g.lda = n; g.B = dM; g.ldb = n; g.C = dR; g.ldc = n;
    g.map = MAP_TRI; g.tiles_m = g.tiles_m_last = T; g.tiles_n = T;
    g.klo_sel = KSEL_TI; g.klo_c = 0; g.khi_sel = KSEL_CONST; g.khi_c = T;
    CHECK(launch_gemm(g, false, false, 1, 0));
    CHECK(cudaDeviceSynchronize());
    std::vector<double> C((size_t)n * n), R((size_t)n * n);
    CHECK(cudaMemcpy(C.data(), dC, sizeof(double) * n * n, cudaMemcpyDeviceToHost));
    CHECK(cudaMemcpy(R.data(), dR, sizeof(double) * n * n, cudaMemcpyDeviceToHost));
    double worst = 0.0, cmax = 0.0;
    for (int i = 0; i < n; i++)
        for (int j = 0; j <= (i / TILE) * TILE + TILE - 1 && j < n; j++) {
            if (j / TILE > i / TILE) continue;
            worst = fmax(worst, fabs(C[(size_t)i * n + j] - R[(size_t)i * n + j]));
            cmax = fmax(cmax, fabs(R[(size_t)i * n + j]));
        }
    printf("lauum shape n=%d: |oz - dmma|max / |dmma|max = %.3e\n", n, worst / cmax);
    if (!(worst / cmax < 1e-13)) fails++;
    fflush(stdout);
    for (int lv = 6; lv >= 5; lv--) {
        // fewer significance levels (the K^-1 product of the engine keeps 6: it only feeds the gradient trace)
        OzGemmOp o2 = op;
        o2.levels = lv;
        CHECK(launch_oz_gemm(tmA, tmB, o2, 1, 0));
        CHECK(cudaDeviceSynchronize());
        CHECK(cudaMemcpy(C.data(), dC, sizeof(double) * n * n, cudaMemcpyDeviceToHost));
        double w2 = 0.0;
        for (int i = 0; i < n; i++)
            for (int j = 0; j < n; j++) {
                if (j / TILE > i / TILE) continue;
                w2 = fmax(w2, fabs(C[(size_t)i * n + j] - R[(size_t)i * n + j]));
            }
        printf("   %d levels: |oz - dmma|max / |dmma|max = %.3e\n", lv, w2 / cmax);
        if (!(w2 / cmax < (lv == 6 ? 1e-10 : 1e-8))) fails++;
    }
    cudaFree(dM); cudaFree(dC); cudaFree(dR);
    free_planes(P);
    return fails;
}

// batched rectangular products with per-entry strides (trtri level shape): C_z = A_z B_z^T, z = 0..nb-1, blocks on
// the diagonal of an n x n matrix
static int check_batched() {
    int fails = 0;
    const int n = 1024, hb = 2, nb = 2;   // two groups of 2*hb tiles: A_z = X[(z*4+2)*128 .. +256, z*512 .. +256]
    std::vector<double> Xh((size_t)n * n), Yh((size_t)n * n);
    unsigned long long seed = 99;
    for (auto& v : Xh) v = urand(seed);
    for (auto& v : Yh) v = urand(seed);
    double *dX, *dY, *dC, *dR;
    CHECK(cudaMalloc(&dX, sizeof(double) * n * n));
    CHECK(cudaMalloc(&dY, sizeof(double) * n * n));
    CHECK(cudaMalloc(&dC, sizeof(double) * n * n));
    CHECK(cudaMalloc(&dR, sizeof(double) * n * n));
    CHECK(cudaMemcpy(dX, Xh.data(), sizeof(double) * n * n, cudaMemcpyHostToDevice));
    CHECK(cudaMemcpy(dY, Yh.data(), sizeof(double) * n * n, cudaMemcpyHostToDevice));
    CHECK(cudaMemset(dC, 0, sizeof(double) * n * n));
    CHECK(cudaMemset(dR, 0, sizeof(double) * n * n));
    OzPlanes PX = alloc_planes(n, n), PY = alloc_planes(n, n);
    const long long zs = (long long)2 * hb * TILE * n + (long long)2 * hb * TILE;   // next group, diagonal step
    const long long off21 = (long long)hb * TILE * n;
    // A_z = X21 block (k-contiguous), B_z = Y11 block given as [k][c] (row-contiguous) -> transposed planes
    CHECK(oz_split_rows(dX + off21, n, zs, hb * TILE, hb * TILE, hb * TILE, PX, hb * TILE, 0, 2 * hb * TILE, 2 * hb * TILE, nb, 0));
    CHECK(oz_split_cols(dY, n, zs, hb * TILE, hb * TILE, hb * TILE, 0, PY, 0, 0, 2 * hb * TILE, 2 * hb * TILE, nb, 0));
    CUtensorMap tmA, tmB;
    CHECK(oz_make_map(&tmA, PX.planes, n, (long long)OZ_S * n, n, OZ_BM));
    CHECK(oz_make_map(&tmB, PY.planes, n, (long long)OZ_S * n, n, OZ_BN));
    OzGemmOp op = oz_default();
    op.a_plane_rows = op.b_plane_rows = n;
    op.a_row0 = hb * TILE; op.a_k0 = 0; op.a_zs_row = 2 * hb * TILE; op.a_zs_k = 2 * hb * TILE;
    op.b_row0 = 0; op.b_k0 = 0; op.b_zs_row = 2 * hb * TILE; op.b_zs_k = 2 * hb * TILE;
    op.a_scale = PX.scale; op.b_scale = PY.scale;
    op.C = dC + off21; op.ldc = n; op.c_zs = zs;
    op.tiles_m = op.tiles_m_last = hb; op.tiles_n = hb;
    op.klo_sel = KSEL_TJ; op.klo_c = 0; op.khi_sel = KSEL_CONST; op.khi_c = hb;
    CHECK(launch_oz_gemm(tmA, tmB, op, nb, 0));
    GemmOp g = gemm_default();
    g.A = dX + off21; g.lda = n; g.a_zs = zs; g.B = dY; g.ldb = n; g.b_zs = zs; g.C = dR + off21; g.ldc = n; g.c_zs = zs;
    g.tiles_m = g.tiles_m_last = hb; g.tiles_n = hb;
    g.klo_sel = KSEL_TJ; g.klo_c = 0; g.khi_sel = KSEL_CONST; g.khi_c = hb;
    CHECK(launch_gemm(g, true, false, nb, 0));
    CHECK(cudaDeviceSynchronize());
    std::vector<double> C((size_t)n * n), R((size_t)n * n);
    CHECK(cudaMemcpy(C.data(), dC, sizeof(double) * n * n, cudaMemcpyDeviceToHost));
    CHECK(cudaMemcpy(R.data(), dR, sizeof(double) * n * n, cudaMemcpyDeviceToHost));
    double worst = 0.0, cmax = 0.0;
    for (size_t i = 0; i < C.size(); i++) {
        worst = fmax(worst, fabs(C[i] - R[i]));
        cmax = fmax(cmax, fabs(R[i]));
    }
    printf("batched KSEL_TJ shape: |oz - dmma|max / |dmma|max = %.3e (|dmma|max %.3e)\n", worst / cmax, cmax);
    if (!(worst / cmax < 1e-13) || !(cmax > 0.0)) fails++;
    fflush(stdout);
    cudaFree(dX); cudaFree(dY); cudaFree(dC); cudaFree(dR);
    free_planes(PX); free_planes(PY);
    return fails;
}

// ---- check groups ---------------------------------------------------------------------------------------------
// Operand entries of the product checks have magnitudes in [0.5, 1] (random sign), so that even a one-term sum is far
// above the representation error of its row: every product check can then use 1e-15 of sum |a||b| (plus |beta C|).
static double mag_rand(unsigned long long& s) {
    const double u = urand(s);
    return (u < 0.0 ? -1.0 : 1.0) * (0.5 + 0.5 * fabs(u));
}
// C outside the live region of a launch is filled with this NaN bit pattern and must come back bit for bit
static const unsigned long long kSentinel = 0x7ff4deadbeef0001ull;
static double sentinel() {
    double d;
    memcpy(&d, &kSentinel, sizeof(d));
    return d;
}
static bool same_bits(double a, double b) { return memcmp(&a, &b, sizeof(double)) == 0; }

static int report(const char* group, const char* what, double err, double bound) {
    const bool ok = err <= bound;   // a NaN error fails
    printf("%s %s: error %.3e bound %.3e %s\n", group, what, err, bound, ok ? "ok" : "FAILED");
    fflush(stdout);
    return ok ? 0 : 1;
}
static int report_count(const char* group, const char* what, long long bad) {
    printf("%s %s: %lld (bound 0) %s\n", group, what, bad, bad ? "FAILED" : "ok");
    fflush(stdout);
    return bad ? 1 : 0;
}
static int group_end(const char* group, int fails) {
    printf("%s: %s (%d failing checks)\n", group, fails ? "FAILED" : "ok", fails);
    fflush(stdout);
    return fails;
}

template <typename Tv>
static Tv* dev_upload(const std::vector<Tv>& h) {
    Tv* d;
    CHECK(cudaMalloc(&d, sizeof(Tv) * h.size()));
    CHECK(cudaMemcpy(d, h.data(), sizeof(Tv) * h.size(), cudaMemcpyHostToDevice));
    return d;
}
template <typename Tv>
static void dev_download(std::vector<Tv>& h, const Tv* d) {
    CHECK(cudaMemcpy(h.data(), d, sizeof(Tv) * h.size(), cudaMemcpyDeviceToHost));
}

// plane buffers of a context hold stale digits of earlier launches in practice: a K range that reaches past the
// region a launch split would pick these up
static void poison_planes(OzCtx& oz) {
    for (OzPlanes* P : {&oz.PP, &oz.PA, &oz.PB, &oz.PW[0], &oz.PW[1]})
        CHECK(cudaMemset(P->planes, 0x3c, (size_t)OZ_S * P->rows * P->pitch));
}

// one level of the recursive-doubling inverse (oz_trtri_level), nb = 3 groups, the last with last_s2 tile rows.
// M is lower triangular by element inside its diagonal tiles and carries data of the same magnitude in the tiles
// above the diagonal, which the K ranges (KSEL_TJ lower bound of part 1, KSEL_TI upper bound of part 2) must exclude.
static int ragged_case(int hb, int T) {
    const char* G = "ragged";
    int fails = 0;
    const int n = T * TILE, h = hb * TILE;
    int nb = 0, last_s2 = 0;
    for (int g = 0;; g++) {   // groups with a non-empty second half (trtri_level)
        int s2 = T - (g * 2 * hb + hb);
        if (s2 <= 0) break;
        nb++;
        last_s2 = s2 < hb ? s2 : hb;
    }
    std::vector<double> L((size_t)n * n), M((size_t)n * n), X((size_t)n * n, sentinel());
    unsigned long long seed = 4242 + T;
    for (auto& v : L) v = mag_rand(seed);
    for (int r = 0; r < n; r++)
        for (int c = 0; c < n; c++) M[(size_t)r * n + c] = (r / TILE == c / TILE && c > r) ? 0.0 : mag_rand(seed);
    double *dL = dev_upload(L), *dM = dev_upload(M), *dX = dev_upload(X);
    OzCtx oz;
    CHECK(oz.init(n));
    poison_planes(oz);
    CHECK(oz_trtri_level(oz, dL, dM, dX, n, hb, 0, nb, last_s2, 1, 0));
    CHECK(cudaDeviceSynchronize());
    std::vector<double> Xg((size_t)n * n), Mg((size_t)n * n);
    dev_download(Xg, dX);
    // part 1: X21 = L21 M11, k blocks [tj, hb) of the group
    double worst = 0.0;
    long long touched = 0;
    std::vector<char> live((size_t)n * n, 0);
    for (int z = 0; z < nb; z++) {
        const int g0 = z * 2 * h, rows = (z == nb - 1 ? last_s2 : hb) * TILE;
        for (int i = g0 + h; i < g0 + h + rows; i++)
            for (int j = g0; j < g0 + h; j++) {
                live[(size_t)i * n + j] = 1;
                long double acc = 0.0L, mag = 0.0L;
                for (int k = g0 + ((j - g0) / TILE) * TILE; k < g0 + h; k++) {
                    const long double t = (long double)L[(size_t)i * n + k] * M[(size_t)k * n + j];
                    acc += t;
                    mag += fabsl(t);
                }
                worst = fmax(worst, (double)(fabsl(Xg[(size_t)i * n + j] - acc) / mag));
            }
    }
    for (size_t e = 0; e < X.size(); e++)
        if (!live[e] && !same_bits(Xg[e], X[e])) touched++;
    char what[160];
    snprintf(what, sizeof(what), "hb=%d T=%d nb=%d last=%d part 1 (X21 = L21 M11) / sum|a||b|", hb, T, nb, last_s2);
    fails += report(G, what, worst, 1e-15);
    snprintf(what, sizeof(what), "hb=%d T=%d part 1 entries changed outside the live X21 blocks", hb, T);
    fails += report_count(G, what, touched);
    // part 2: M21 = -M22 X21, k blocks [0, ti] of the group's second half (X21 as computed above).  X21 is a computed
    // operand: its entries cancel to far below their column maximum, which sets the column's scale, so the error is
    // measured against sum_k |M22[i,k]| max_k' |X21[k',j]| (the representation error of a column is <= its scale 2^-56)
    CHECK(oz_trtri_level(oz, dL, dM, dX, n, hb, 0, nb, last_s2, 2, 0));
    CHECK(cudaDeviceSynchronize());
    dev_download(Mg, dM);
    worst = 0.0;
    touched = 0;
    for (int z = 0; z < nb; z++) {
        const int g0 = z * 2 * h, rows = (z == nb - 1 ? last_s2 : hb) * TILE;
        std::vector<double> colmax(h, 0.0);
        for (int k = g0 + h; k < g0 + h + rows; k++)
            for (int j = g0; j < g0 + h; j++) colmax[j - g0] = fmax(colmax[j - g0], fabs(Xg[(size_t)k * n + j]));
        for (int i = g0 + h; i < g0 + h + rows; i++)
            for (int j = g0; j < g0 + h; j++) {
                long double acc = 0.0L, mag = 0.0L;
                const int kend = g0 + h + ((i - g0 - h) / TILE + 1) * TILE;
                for (int k = g0 + h; k < kend; k++) {
                    acc -= (long double)M[(size_t)i * n + k] * Xg[(size_t)k * n + j];
                    mag += fabsl((long double)M[(size_t)i * n + k]) * colmax[j - g0];
                }
                worst = fmax(worst, (double)(fabsl(Mg[(size_t)i * n + j] - acc) / mag));
            }
    }
    for (size_t e = 0; e < M.size(); e++)
        if (!live[e] && !same_bits(Mg[e], M[e])) touched++;
    snprintf(what, sizeof(what), "hb=%d T=%d nb=%d last=%d part 2 (M21 = -M22 X21) / sum|a| max|b|", hb, T, nb, last_s2);
    fails += report(G, what, worst, 1e-15);
    snprintf(what, sizeof(what), "hb=%d T=%d part 2 entries of M changed outside the live M21 blocks", hb, T);
    fails += report_count(G, what, touched);
    oz.destroy();
    cudaFree(dL); cudaFree(dM); cudaFree(dX);
    return fails;
}

static int check_ragged() {
    int fails = 0;
    fails += ragged_case(4, 21);   // groups of 8 tiles: 2 full, the last with 1 tile row
    fails += ragged_case(4, 23);   // the last with hb - 1 = 3 tile rows
    return group_end("ragged", fails);
}

static int check_maps() {
    const char* G = "maps";
    int fails = 0;
    const int T = 10, n = T * TILE;
    unsigned long long seed = 515;
    OzCtx oz;
    CHECK(oz.init(n));
    poison_planes(oz);
    {
        // C[i,j] -= sum_{k in panel [0,2)} A[i,k] A[j,k] on tile rows [4,10) x tile columns [2,8), i >= j:
        // lower_filter with lower_off = 2 (tiles (4,5..7), (5,6..7), (6,7) are filtered out)
        const int p0 = 0, pend = 2, r0 = 4, r1 = 10, c0 = 2, c1 = 8;
        std::vector<double> A((size_t)n * n);
        for (auto& v : A) v = mag_rand(seed);
        double* dA = dev_upload(A);
        CHECK(oz_split_panel_rows(oz, dA, n, p0, pend, c0, r1, 0, 0));
        CHECK(oz_update_region(oz, dA, n, p0, pend, r0, r1, c0, c1, 0, 0));
        CHECK(cudaDeviceSynchronize());
        std::vector<double> Ag((size_t)n * n);
        dev_download(Ag, dA);
        double worst = 0.0;
        long long touched = 0;
        for (int i = 0; i < n; i++)
            for (int j = 0; j < n; j++) {
                const int ti = i / TILE, tj = j / TILE;
                const bool in = ti >= r0 && ti < r1 && tj >= c0 && tj < c1 && ti >= tj;
                if (!in) {
                    if (!same_bits(Ag[(size_t)i * n + j], A[(size_t)i * n + j])) touched++;
                    continue;
                }
                long double acc = A[(size_t)i * n + j], mag = fabs(A[(size_t)i * n + j]);
                for (int k = p0 * TILE; k < pend * TILE; k++) {
                    const long double t = (long double)A[(size_t)i * n + k] * A[(size_t)j * n + k];
                    acc -= t;
                    mag += fabsl(t);
                }
                worst = fmax(worst, (double)(fabsl(Ag[(size_t)i * n + j] - acc) / mag));
            }
        fails += report(G, "oz_update_region rows [4,10) x cols [2,8) lower_off 2, alpha -1 beta 1 / (|C| + sum|a||b|)",
                        worst, 1e-15);
        fails += report_count(G, "oz_update_region entries changed outside the live tiles (filtered tiles included)", touched);
        cudaFree(dA);
    }
    {
        // lazy panel solve X = A W^T in place on rows [5,10) x panel columns [2,5): k blocks [0, tj]; W lower triangular
        // by element in its diagonal tiles, data of the same magnitude in the tiles above (excluded by KSEL_TJ)
        const int p0 = 2, pend = 5, pw = pend - p0, r0 = 5, r1 = 10;
        std::vector<double> A((size_t)n * n), W((size_t)n * n, 0.0);
        for (auto& v : A) v = mag_rand(seed);
        for (int r = 0; r < pw * TILE; r++)
            for (int c = 0; c < pw * TILE; c++)
                W[(size_t)r * n + c] = (r / TILE == c / TILE && c > r) ? 0.0 : mag_rand(seed);
        double *dA = dev_upload(A), *dW = dev_upload(W);
        CHECK(oz_split_w(oz, dW, n, pw, 1, 0));
        CHECK(oz_panel_solve(oz, dA, n, p0, pend, r0, r1, 1, 4, 0));
        CHECK(cudaDeviceSynchronize());
        std::vector<double> Ag((size_t)n * n);
        dev_download(Ag, dA);
        double worst = 0.0;
        long long touched = 0;
        for (int i = 0; i < n; i++)
            for (int j = 0; j < n; j++) {
                const int ti = i / TILE, tj = j / TILE;
                if (!(ti >= r0 && ti < r1 && tj >= p0 && tj < pend)) {
                    if (!same_bits(Ag[(size_t)i * n + j], A[(size_t)i * n + j])) touched++;
                    continue;
                }
                const int c = j - p0 * TILE;
                long double acc = 0.0L, mag = 0.0L;
                for (int k = 0; k < (c / TILE + 1) * TILE; k++) {
                    const long double t = (long double)A[(size_t)i * n + p0 * TILE + k] * W[(size_t)c * n + k];
                    acc += t;
                    mag += fabsl(t);
                }
                worst = fmax(worst, (double)(fabsl(Ag[(size_t)i * n + j] - acc) / mag));
            }
        fails += report(G, "oz_panel_solve rows [5,10) x panel [2,5), B planes of LAZY_PB*128 rows / sum|a||b|", worst, 1e-15);
        fails += report_count(G, "oz_panel_solve entries changed outside the panel rows", touched);
        cudaFree(dA);
        cudaFree(dW);
    }
    oz.destroy();
    return group_end(G, fails);
}

// K range of S = 2 * 128 + 10 blocks cut into k_min / k_max segments of <= 128 blocks (beta 0, then 1), as oz_lauum
// does for N > 16384.  Item (ti, tj) accumulates k blocks [127 + ti, 255 + tj): item row 1 has an empty range in the
// first segment (C <- 0 C), item columns 0 and 1 in the last (C <- C).
static int check_segments() {
    const char* G = "segments";
    int fails = 0;
    const int S = 2 * 128 + 10, K = S * TILE, m = 2 * TILE, nc = 3 * TILE;
    unsigned long long seed = 266;
    std::vector<double> A((size_t)m * K), B((size_t)nc * K);
    for (auto& v : A) v = mag_rand(seed);
    for (auto& v : B) v = mag_rand(seed);
    double *dA = dev_upload(A), *dB = dev_upload(B);
    std::vector<double> C((size_t)m * nc, sentinel());
    double* dC = dev_upload(C);
    OzPlanes PA = alloc_planes(m, K), PB = alloc_planes(nc, K);
    CHECK(oz_split_rows(dA, K, 0, m, m, K, PA, 0, 0, 0, 0, 1, 0));
    CHECK(oz_split_rows(dB, K, 0, nc, nc, K, PB, 0, 0, 0, 0, 1, 0));
    CUtensorMap tmA, tmB;
    CHECK(oz_make_map(&tmA, PA.planes, K, (long long)OZ_S * m, K, OZ_BM));
    CHECK(oz_make_map(&tmB, PB.planes, K, (long long)OZ_S * nc, K, OZ_BN));
    OzGemmOp op = oz_default();
    op.a_plane_rows = m;
    op.b_plane_rows = nc;
    op.a_scale = PA.scale;
    op.b_scale = PB.scale;
    op.C = dC;
    op.ldc = nc;
    op.tiles_m = op.tiles_m_last = m / TILE;
    op.tiles_n = nc / TILE;
    op.klo_sel = KSEL_TI;
    op.klo_c = 127;
    op.khi_sel = KSEL_TJ;
    op.khi_c = 255;
    for (int k0 = 0; k0 < S; k0 += 128) {
        op.k_min = k0;
        op.k_max = std::min(k0 + 128, S);
        op.beta = k0 == 0 ? 0.0 : 1.0;
        CHECK(launch_oz_gemm(tmA, tmB, op, 1, 0));
    }
    CHECK(cudaDeviceSynchronize());
    dev_download(C, dC);
    double worst = 0.0;
    long long nonfinite = 0;
    for (int i = 0; i < m; i++)
        for (int j = 0; j < nc; j++) {
            if (!isfinite(C[(size_t)i * nc + j])) {   // e.g. the sentinel carried through the C <- 0 C path
                nonfinite++;
                continue;
            }
            long double acc = 0.0L, mag = 0.0L;
            for (int k = (127 + i / TILE) * TILE; k < (255 + j / TILE) * TILE; k++) {
                const long double t = (long double)A[(size_t)i * K + k] * B[(size_t)j * K + k];
                acc += t;
                mag += fabsl(t);
            }
            worst = fmax(worst, (double)(fabsl(C[(size_t)i * nc + j] - acc) / mag));
        }
    // ~17000 terms of random sign per entry: representation errors and FP64 roundings average out (observed ~5e-18 of
    // sum |a||b|), so the bound is 1e-16 here; with 6 instead of 7 significance levels the error is ~8e-16
    fails += report(G, "K range of 266 blocks in 3 segments (empty ranges included) / sum|a||b|", worst, 1e-16);
    fails += report_count(G, "non-finite entries of C (sentinel NaN before the first segment)", nonfinite);
    cudaFree(dA); cudaFree(dB); cudaFree(dC);
    free_planes(PA); free_planes(PB);
    return group_end(G, fails);
}

// digit planes written directly (not through a split): K = 16384 (128 blocks, the longest single accumulation)
static int check_limits() {
    const char* G = "limits";
    int fails = 0;
    const int K = 128 * TILE;
    {
        // d_0 = -64, d_1..6 = -128 in both operands: every pair product is positive; level 6 sums
        // 2 * 64 * 128 + 5 * 128 * 128 = 98304 per k, 1.61e9 over K (int32 limit 2.15e9)
        const int m = TILE;
        OzPlanes PA = alloc_planes(m, K), PB = alloc_planes(m, K);
        for (OzPlanes* P : {&PA, &PB}) {
            CHECK(cudaMemset(P->planes, 0xc0, (size_t)m * K));                        // plane 0: -64
            CHECK(cudaMemset(P->planes + (size_t)m * K, 0x80, (size_t)(OZ_S - 1) * m * K));   // planes 1..6: -128
            std::vector<double> one(m, 1.0);
            CHECK(cudaMemcpy(P->scale, one.data(), sizeof(double) * m, cudaMemcpyHostToDevice));
        }
        double* dC;
        CHECK(cudaMalloc(&dC, sizeof(double) * m * m));
        CUtensorMap tmA, tmB;
        CHECK(oz_make_map(&tmA, PA.planes, K, (long long)OZ_S * m, K, OZ_BM));
        CHECK(oz_make_map(&tmB, PB.planes, K, (long long)OZ_S * m, K, OZ_BN));
        OzGemmOp op = oz_default();
        op.a_plane_rows = op.b_plane_rows = m;
        op.a_scale = PA.scale;
        op.b_scale = PB.scale;
        op.C = dC;
        op.ldc = m;
        op.tiles_m = op.tiles_m_last = 1;
        op.tiles_n = 1;
        op.khi_c = 128;
        CHECK(launch_oz_gemm(tmA, tmB, op, 1, 0));
        CHECK(cudaDeviceSynchronize());
        std::vector<double> C((size_t)m * m);
        dev_download(C, dC);
        const long long d[OZ_S] = {-64, -128, -128, -128, -128, -128, -128};
        long long lv[OZ_S] = {0};
        for (int i = 0; i < OZ_S; i++)
            for (int j = 0; i + j < OZ_S; j++) lv[i + j] += d[i] * d[j] * (long long)K;
        long double want = 0.0L;
        for (int l = OZ_S - 1; l >= 0; l--) want = want / 256.0L + (long double)lv[l];
        want /= 65536.0L;
        double worst = 0.0;
        for (double v : C) worst = fmax(worst, (double)(fabsl(v - want) / want));
        printf("%s largest accumulation: level 6 sums %lld (int32 limit %d)\n", G, lv[OZ_S - 1], 2147483647);
        fails += report(G, "extreme digits, K = 16384, against the closed form / value", worst, ldexp(1.0, -52));
        cudaFree(dC);
        free_planes(PA); free_planes(PB);
    }
    {
        // random digits (|d_0| <= 64) and power-of-two scales, 7 / 6 / 5 levels against int64 host sums over the
        // same levels at 400 sampled entries
        const int m = 2 * TILE;
        std::vector<int8_t> a((size_t)OZ_S * m * K), b((size_t)OZ_S * m * K);
        std::vector<double> sa(m), sb(m);
        unsigned long long seed = 16384;
        for (auto* v : {&a, &b})
            for (size_t e = 0; e < v->size(); e++) {
                seed = seed * 6364136223846793005ull + 1442695040888963407ull;
                const int r = (int)(seed >> 33);
                (*v)[e] = e < (size_t)m * K ? (int8_t)(r % 129 - 64) : (int8_t)(r & 0xff);
            }
        for (int r = 0; r < m; r++) {
            sa[r] = ldexp(1.0, (int)(8.0 * urand(seed)));
            sb[r] = ldexp(1.0, (int)(8.0 * urand(seed)));
        }
        OzPlanes PA = alloc_planes(m, K), PB = alloc_planes(m, K);
        CHECK(cudaMemcpy(PA.planes, a.data(), a.size(), cudaMemcpyHostToDevice));
        CHECK(cudaMemcpy(PB.planes, b.data(), b.size(), cudaMemcpyHostToDevice));
        CHECK(cudaMemcpy(PA.scale, sa.data(), sizeof(double) * m, cudaMemcpyHostToDevice));
        CHECK(cudaMemcpy(PB.scale, sb.data(), sizeof(double) * m, cudaMemcpyHostToDevice));
        double* dC;
        CHECK(cudaMalloc(&dC, sizeof(double) * m * m));
        CUtensorMap tmA, tmB;
        CHECK(oz_make_map(&tmA, PA.planes, K, (long long)OZ_S * m, K, OZ_BM));
        CHECK(oz_make_map(&tmB, PB.planes, K, (long long)OZ_S * m, K, OZ_BN));
        const int ns = 400;
        std::vector<int> si(ns), sj(ns);
        std::vector<long long> lv((size_t)ns * OZ_S, 0);
        for (int s = 0; s < ns; s++) {
            si[s] = (int)((urand(seed) * 0.5 + 0.5) * m) % m;
            sj[s] = (int)((urand(seed) * 0.5 + 0.5) * m) % m;
            for (int i = 0; i < OZ_S; i++)
                for (int j = 0; i + j < OZ_S; j++) {
                    const int8_t* pa = &a[((size_t)i * m + si[s]) * K];
                    const int8_t* pb = &b[((size_t)j * m + sj[s]) * K];
                    long long acc = 0;
                    for (int k = 0; k < K; k++) acc += (long long)pa[k] * pb[k];
                    lv[(size_t)s * OZ_S + i + j] += acc;
                }
        }
        std::vector<double> C((size_t)m * m);
        for (int levels : {7, 6, 5}) {
            OzGemmOp op = oz_default();
            op.a_plane_rows = op.b_plane_rows = m;
            op.a_scale = PA.scale;
            op.b_scale = PB.scale;
            op.C = dC;
            op.ldc = m;
            op.tiles_m = op.tiles_m_last = m / TILE;
            op.tiles_n = m / TILE;
            op.khi_c = 128;
            op.levels = levels == 7 ? 0 : levels;
            CHECK(launch_oz_gemm(tmA, tmB, op, 1, 0));
            CHECK(cudaDeviceSynchronize());
            dev_download(C, dC);
            double worst = 0.0;
            for (int s = 0; s < ns; s++) {
                long double want = 0.0L, mag = 0.0L;
                for (int l = levels - 1; l >= 0; l--) {
                    want = want / 256.0L + (long double)lv[(size_t)s * OZ_S + l];
                    mag = mag / 256.0L + fabsl((long double)lv[(size_t)s * OZ_S + l]);
                }
                const long double sc = (long double)sa[si[s]] * sb[sj[s]] / 65536.0L;
                worst = fmax(worst, (double)(fabsl(C[(size_t)si[s] * m + sj[s]] - want * sc) / (mag * sc)));
            }
            char what[160];
            snprintf(what, sizeof(what), "random digits, K = 16384, %d levels, 400 entries against int64 sums / magnitude", levels);
            fails += report(G, what, worst, ldexp(1.0, -52));
        }
        cudaFree(dC);
        free_planes(PA); free_planes(PB);
    }
    return group_end(G, fails);
}

// the documented split of one row: scale 2^(ex+2) for a finite non-zero maximum below 1e300, else scale 1 and zero digits
static double host_scale(double amax, bool& zero_digits) {
    zero_digits = !(amax > 0.0) || !(amax < 1.0e300);
    if (zero_digits) return 1.0;
    int ex;
    frexp(amax, &ex);
    return ldexp(1.0, ex + 2);
}

static int check_exponents() {
    const char* G = "exponents";
    int fails = 0;
    const int R = 256, K = 128, NB = 128;
    std::vector<double> X((size_t)R * K, 0.0);
    unsigned long long seed = 1074;
    auto row = [&](int r) { return &X[(size_t)r * K]; };
    // rows 1..199: maxima swept over 2^-1074 .. 2^996 (entries of magnitude [0.5, 1] x 2^e and some smaller)
    for (int r = 1; r < 200; r++) {
        const int e = -1074 + (int)((long long)(r - 1) * (996 + 1074) / 198);
        for (int k = 0; k < K; k++) row(r)[k] = ldexp(mag_rand(seed) * ((k % 5 == 0) ? 1e-3 : 1.0), e);
    }
    // rows 200..223: exact powers of two of both signs, around the 2^-970 boundary and at both ends
    const int pw[12] = {-1074, -1073, -1060, -1022, -1000, -971, -970, -969, -500, 0, 995, 996};
    for (int q = 0; q < 24; q++) {
        const int r = 200 + q, e = pw[q % 12];
        for (int k = 0; k < K; k++) row(r)[k] = ldexp((q < 12) == (k % 2 == 0) ? 1.0 : -1.0, e - (k % 3));
    }
    // rows 224..235: a single non-zero entry
    for (int q = 0; q < 12; q++) row(224 + q)[(q * 37) % K] = ldexp(mag_rand(seed), pw[q]);
    // rows 236..247: subnormal entries next to normal maxima (and one all-subnormal row)
    for (int q = 0; q < 12; q++) {
        const int r = 236 + q, e = q == 11 ? -1040 : -1022 + 6 * q;
        for (int k = 0; k < K; k++) row(r)[k] = ldexp(mag_rand(seed), k == 3 ? e : -1050 - (k % 20));
    }
    // rows 248..251 NaN (every entry), 252 / 253 one +Inf / -Inf entry, 0 and 254..255 zero
    for (int r = 248; r < 252; r++)
        for (int k = 0; k < K; k++) row(r)[k] = nan("");
    row(252)[5] = INFINITY;
    row(253)[77] = -INFINITY;
    std::vector<double> Xt((size_t)K * R);
    for (int r = 0; r < R; r++)
        for (int k = 0; k < K; k++) Xt[(size_t)k * R + r] = X[(size_t)r * K + k];
    double *dX = dev_upload(X), *dXt = dev_upload(Xt);
    OzPlanes PR = alloc_planes(R, K), PC = alloc_planes(R, K);
    CHECK(oz_split_rows(dX, K, 0, R, R, K, PR, 0, 0, 0, 0, 1, 0));
    CHECK(oz_split_cols(dXt, R, 0, K, K, R, 0, PC, 0, 0, 0, 0, 1, 0));
    CHECK(cudaDeviceSynchronize());
    std::vector<int8_t> hr((size_t)OZ_S * R * K), hc((size_t)OZ_S * R * K);
    std::vector<double> sr(R), sc(R);
    dev_download(hr, PR.planes);
    dev_download(hc, PC.planes);
    dev_download(sr, PR.scale);
    dev_download(sc, PC.scale);
    long long bad_rows = 0, bad_cols = 0, bad_tiny = 0;
    double worst_rep = 0.0;
    for (int r = 0; r < R; r++) {
        double amax = 0.0;
        for (int k = 0; k < K; k++) amax = fmax(amax, fabs(row(r)[k]));   // fmax drops NaN, as on the device
        bool zero;
        const double s = host_scale(amax, zero);
        bool row_bad = !same_bits(sr[r], s), col_bad = !same_bits(sc[r], s);
        for (int k = 0; k < K; k++) {
            int8_t d[OZ_S] = {0, 0, 0, 0, 0, 0, 0};
            if (!zero) host_digits(row(r)[k], s, d);
            long double rep = 0.0L;
            for (int p = 0; p < OZ_S; p++) {
                const int8_t g = hr[((size_t)p * R + r) * K + k];
                row_bad |= g != d[p];
                col_bad |= hc[((size_t)p * R + r) * K + k] != d[p];
                rep += (long double)g * powl(256.0L, -(p + 1));
            }
            if (!zero) {
                // documented: x = scale * sum_p d_p 256^-(p+1) + t, 0 <= t < scale 2^-56
                const long double t = ((long double)row(r)[k] - rep * s) / s;
                worst_rep = fmax(worst_rep, t < 0 ? 1.0 : (double)t);
            }
        }
        bad_rows += row_bad;
        bad_cols += col_bad;
        if ((row_bad || col_bad) && amax > 0.0 && amax < ldexp(1.0, -970)) bad_tiny++;
    }
    printf("%s rows with a maximum below 2^-970 among the mismatching rows: %lld\n", G, bad_tiny);
    fails += report_count(G, "split_rows rows whose scale or digits differ from the documented split", bad_rows);
    fails += report_count(G, "split_cols rows whose scale or digits differ from the documented split", bad_cols);
    fails += report(G, "representation t / scale on every finite row (bound 2^-56, t >= 0)", worst_rep, ldexp(1.0, -56));
    // product of these rows with moderate ones: 1e-15 of sum |a||b| plus an absolute floor (the scale products of the
    // smallest rows are subnormal or zero); NaN / Inf rows are excluded (their planes are zero by contract)
    std::vector<double> B((size_t)NB * K);
    for (int c = 0; c < NB; c++) {
        const int e = -(int)(20.0 * (urand(seed) * 0.5 + 0.5));
        for (int k = 0; k < K; k++) B[(size_t)c * K + k] = ldexp(mag_rand(seed), e);
    }
    double* dB = dev_upload(B);
    OzPlanes PB = alloc_planes(NB, K);
    CHECK(oz_split_rows(dB, K, 0, NB, NB, K, PB, 0, 0, 0, 0, 1, 0));
    double* dC;
    CHECK(cudaMalloc(&dC, sizeof(double) * R * NB));
    CUtensorMap tmA, tmB;
    CHECK(oz_make_map(&tmA, PR.planes, K, (long long)OZ_S * R, K, OZ_BM));
    CHECK(oz_make_map(&tmB, PB.planes, K, (long long)OZ_S * NB, K, OZ_BN));
    OzGemmOp op = oz_default();
    op.a_plane_rows = R;
    op.b_plane_rows = NB;
    op.a_scale = PR.scale;
    op.b_scale = PB.scale;
    op.C = dC;
    op.ldc = NB;
    op.tiles_m = op.tiles_m_last = R / TILE;
    op.tiles_n = NB / TILE;
    op.khi_c = K / TILE;
    CHECK(launch_oz_gemm(tmA, tmB, op, 1, 0));
    CHECK(cudaDeviceSynchronize());
    std::vector<double> C((size_t)R * NB);
    dev_download(C, dC);
    const double floor_abs = ldexp(1.0, -1000);
    double worst = 0.0;
    for (int r = 0; r < R; r++) {
        if (r >= 248 && r <= 253) continue;
        for (int c = 0; c < NB; c++) {
            long double acc = 0.0L, mag = 0.0L;
            for (int k = 0; k < K; k++) {
                const long double t = (long double)row(r)[k] * B[(size_t)c * K + k];
                acc += t;
                mag += fabsl(t);
            }
            worst = fmax(worst, (double)(fabsl(C[(size_t)r * NB + c] - acc) / (1e-15L * mag + floor_abs)));
        }
    }
    fails += report(G, "product of the finite rows, |error| / (1e-15 sum|a||b| + 2^-1000)", worst, 1.0);
    cudaFree(dX); cudaFree(dXt); cudaFree(dB); cudaFree(dC);
    free_planes(PR); free_planes(PC); free_planes(PB);
    return group_end(G, fails);
}

__global__ void fill_rand(double* A, long long n, unsigned seed) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    unsigned long long s = (unsigned long long)i * 2654435761ull + seed;
    s ^= s >> 17; s *= 0xed5ad4bbull; s ^= s >> 11; s *= 0xac4c1b51ull; s ^= s >> 15;
    A[i] = ((double)(s & 0xffffffffull) / 4294967296.0) * 2.0 - 1.0;
}

static void perf(int n, int kblocks, int tri, int reps) {
    // C (n x n, or lower tiles) = A[:, :K] B[:, :K]^T with K = kblocks * 128 (tri: K range [ti, T) like K^-1 = M^T M)
    const int T = n / TILE;
    double *dA, *dC;
    CHECK(cudaMalloc(&dA, sizeof(double) * n * n));
    CHECK(cudaMalloc(&dC, sizeof(double) * n * n));
    fill_rand<<<(unsigned)(((long long)n * n + 255) / 256), 256>>>(dA, (long long)n * n, 7u);
    CHECK(cudaMemset(dC, 0, sizeof(double) * n * n));
    OzPlanes P = alloc_planes(n, n);
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    float ms_split_r = 0, ms_split_c = 0, ms_oz = 0, ms_dmma = 0;
    CHECK(oz_split_rows(dA, n, 0, n, n, kblocks * TILE, P, 0, 0, 0, 0, 1, 0));
    cudaEventRecord(e0);
    for (int i = 0; i < reps; i++) CHECK(oz_split_rows(dA, n, 0, n, n, kblocks * TILE, P, 0, 0, 0, 0, 1, 0));
    cudaEventRecord(e1);
    CHECK(cudaEventSynchronize(e1));
    cudaEventElapsedTime(&ms_split_r, e0, e1);
    ms_split_r /= reps;
    if (kblocks == T) {
        cudaEventRecord(e0);
        for (int i = 0; i < reps; i++) CHECK(oz_split_cols(dA, n, 0, n, n, n, tri, P, 0, 0, 0, 0, 1, 0));
        cudaEventRecord(e1);
        CHECK(cudaEventSynchronize(e1));
        cudaEventElapsedTime(&ms_split_c, e0, e1);
        ms_split_c /= reps;
    }
    CUtensorMap tmA, tmB;
    CHECK(oz_make_map(&tmA, P.planes, n, (long long)OZ_S * n, n, OZ_BM));
    CHECK(oz_make_map(&tmB, P.planes, n, (long long)OZ_S * n, n, OZ_BN));
    OzGemmOp op = oz_default();
    op.a_plane_rows = op.b_plane_rows = n;
    op.a_scale = op.b_scale = P.scale;
    op.C = dC; op.ldc = n;
    op.tiles_m = op.tiles_m_last = T; op.tiles_n = T;
    op.map = MAP_TRI;
    if (tri) { op.klo_sel = KSEL_TI; op.klo_c = 0; op.khi_c = T; }
    else { op.klo_c = 0; op.khi_c = kblocks; op.alpha = -1.0; op.beta = 1.0; }
    CHECK(launch_oz_gemm(tmA, tmB, op, 1, 0));
    CHECK(cudaDeviceSynchronize());
    {
        long long* dprof;
        CHECK(cudaMalloc(&dprof, 8 * sizeof(long long)));
        CHECK(cudaMemset(dprof, 0, 8 * sizeof(long long)));
        OzGemmOp o2 = op;
        o2.prof = dprof;
        CHECK(launch_oz_gemm(tmA, tmB, o2, 1, 0));
        CHECK(cudaDeviceSynchronize());
        long long hp[8];
        CHECK(cudaMemcpy(hp, dprof, sizeof(hp), cudaMemcpyDeviceToHost));
        printf("   CTA 0, first tile (cycles since pass-0 start): p0 issued %lld  complete %lld  epilogue done %lld | p1 start %lld issued %lld"
               " complete %lld epilogue done %lld\n", hp[1] - hp[0], hp[2] - hp[0], hp[3] - hp[0], hp[4] - hp[0], hp[5] - hp[0],
               hp[6] - hp[0], hp[7] - hp[0]);
        cudaFree(dprof);
    }
    cudaEventRecord(e0);
    for (int i = 0; i < reps; i++) CHECK(launch_oz_gemm(tmA, tmB, op, 1, 0));
    cudaEventRecord(e1);
    CHECK(cudaEventSynchronize(e1));
    cudaEventElapsedTime(&ms_oz, e0, e1);
    ms_oz /= reps;
    float ms_lv[2] = {0.f, 0.f};
    if (tri) {
        for (int q = 0; q < 2; q++) {
            OzGemmOp o2 = op;
            o2.levels = 6 - q;
            CHECK(launch_oz_gemm(tmA, tmB, o2, 1, 0));
            cudaEventRecord(e0);
            for (int i = 0; i < reps; i++) CHECK(launch_oz_gemm(tmA, tmB, o2, 1, 0));
            cudaEventRecord(e1);
            CHECK(cudaEventSynchronize(e1));
            cudaEventElapsedTime(&ms_lv[q], e0, e1);
            ms_lv[q] /= reps;
        }
        printf("   K^-1 shape with 6 levels (21 pairs): %.3f ms, 5 levels (15 pairs): %.3f ms\n", ms_lv[0], ms_lv[1]);
    }
    GemmOp g = gemm_default();
    g.A = dA; g.lda = n; g.B = dA; g.ldb = n; g.C = dC; g.ldc = n;
    g.map = MAP_TRI; g.tiles_m = g.tiles_m_last = T; g.tiles_n = T;
    if (tri) { g.klo_sel = KSEL_TI; g.klo_c = 0; g.khi_c = T; }
    else { g.klo_c = 0; g.khi_c = kblocks; g.alpha = -1.0; g.beta = 1.0; }
    CHECK(launch_gemm(g, !tri, !tri, 1, 0));
    CHECK(cudaDeviceSynchronize());
    cudaEventRecord(e0);
    for (int i = 0; i < reps; i++) CHECK(launch_gemm(g, !tri, !tri, 1, 0));
    cudaEventRecord(e1);
    CHECK(cudaEventSynchronize(e1));
    cudaEventElapsedTime(&ms_dmma, e0, e1);
    ms_dmma /= reps;
    // flops: lower tiles x K range
    double flops = 0.0;
    for (int ti = 0; ti < T; ti++)
        for (int tj = 0; tj <= ti; tj++) flops += 2.0 * TILE * TILE * (double)TILE * (tri ? (T - ti) : kblocks);
    printf("n=%d %s K=%d: oz %.3f ms = %.1f TFLOP/s-eq (int8 %.0f TOPS), dmma %.3f ms = %.1f TFLOP/s, split_rows %.3f ms"
           " split_cols %.3f ms\n", n, tri ? "lauum" : "syrk", tri ? n : kblocks * TILE, ms_oz, flops / ms_oz * 1e-9,
           flops * 28.0 / ms_oz * 1e-9, ms_dmma, flops / ms_dmma * 1e-9, ms_split_r, ms_split_c);
    fflush(stdout);
    cudaFree(dA); cudaFree(dC);
    free_planes(P);
}


// ---- raw tcgen05 kind::i8 issue rate: one CTA per SM, MMAs back to back on resident shared-memory tiles ----------
template <int N, int KB>
__global__ void __launch_bounds__(128, 1) mma_rate_kernel(int iters, int a_tiles, int b_tiles, long long* cycles) {
    extern __shared__ uint8_t raw[];
    uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(raw) + 1023) & ~(uintptr_t)1023);
    __shared__ uint64_t bar;
    __shared__ uint32_t slot;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int i = threadIdx.x; i < (a_tiles * 128 * KB + b_tiles * N * KB) / 4; i += blockDim.x) reinterpret_cast<uint32_t*>(base)[i] = 0x01010101u;
    if (threadIdx.x == 0) { mbar_init(&bar, 1); fence_barrier_init(); }
    if (warp == 0) tmem_alloc(&slot, 512);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tm = slot;
    constexpr uint64_t layout = (KB == 128) ? 2 : (KB == 64 ? 4 : 6);
    constexpr uint32_t idesc = (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
    if (warp == 1 && lane == 0) {
        const uint32_t sa = smem_u32(base), sb = sa + a_tiles * 128 * KB;
        const long long t0 = clock64();
        const int nacc = 512 / N;
        const uint64_t hi = ((uint64_t)((8 * KB) >> 4) << 32) | (1ull << 46) | (layout << 61);
        for (int it = 0; it < iters; it += 8) {
#pragma unroll
            for (int u = 0; u < 8; u++) {
                // operand tiles rotate with compile-time offsets; a_tiles / b_tiles are powers of two or 7 (masked to < 8)
                const int ia = (u * 3) % 8 < a_tiles ? (u * 3) % 8 : 0, ib = (u * 5) % 8 < b_tiles ? (u * 5) % 8 : 0;
#pragma unroll
                for (int ks = 0; ks < KB / 32; ks++) {
                    const uint64_t ad = (uint64_t)(((sa + ia * 128 * KB + ks * 32) & 0x3FFFF) >> 4) | hi;
                    const uint64_t bd = (uint64_t)(((sb + ib * N * KB + ks * 32) & 0x3FFFF) >> 4) | hi;
                    umma_i8(tm + (u % nacc) * N, ad, bd, idesc, 1u);
                }
            }
        }
        umma_commit(&bar);
        mbar_wait(&bar, 0);
        const long long t1 = clock64();
        if (blockIdx.x == 0) cycles[0] = t1 - t0;
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tm, 512);
}

template <int N, int KB>
static void mma_rate(int a_tiles, int b_tiles) {
    long long* dc;
    CHECK(cudaMalloc(&dc, 8));
    const int smem = a_tiles * 128 * KB + b_tiles * N * KB + 2048;
    CHECK(cudaFuncSetAttribute(mma_rate_kernel<N, KB>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    const int iters = 8192;
    mma_rate_kernel<N, KB><<<148, 128, smem>>>(iters, a_tiles, b_tiles, dc);
    CHECK(cudaDeviceSynchronize());
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    cudaEventRecord(e0);
    mma_rate_kernel<N, KB><<<148, 128, smem>>>(iters, a_tiles, b_tiles, dc);
    cudaEventRecord(e1);
    CHECK(cudaEventSynchronize(e1));
    float ms; cudaEventElapsedTime(&ms, e0, e1);
    long long cyc; CHECK(cudaMemcpy(&cyc, dc, 8, cudaMemcpyDeviceToHost));
    const double nm = (double)iters * (KB / 32);
    printf("i8 MMA M=128 N=%d (K chunk %d B, %d A tiles, %d B tiles): %.1f cycles per MMA (ideal %.1f), %.0f TOPS on 148 SMs\n", N, KB,
           a_tiles, b_tiles, (double)cyc / nm, 128.0 * N * 32 / 7736.0 * 1.0, 148.0 * nm * 2.0 * 128 * N * 32 / (ms * 1e-3) * 1e-12);
    fflush(stdout);
    cudaFree(dc);
}

int main(int argc, char** argv) {
    const char* what = argc > 1 ? argv[1] : "all";
    int fails = 0;
    CHECK(oz_set_attributes());
    CHECK(gemm_set_attributes());
    if (!strcmp(what, "rate")) {
        mma_rate<64, 64>(7, 7);
        mma_rate<64, 64>(1, 1);
        mma_rate<128, 64>(7, 7);
        mma_rate<128, 64>(1, 1);
        mma_rate<256, 64>(4, 4);
        mma_rate<256, 64>(1, 1);
        mma_rate<64, 128>(4, 4);
        mma_rate<128, 128>(4, 4);
        mma_rate<256, 128>(2, 2);
        mma_rate<64, 32>(7, 7);
        mma_rate<128, 32>(7, 7);
        return 0;
    }
    const struct { const char* name; int (*fn)(); } groups[] = {
        {"ragged", check_ragged}, {"maps", check_maps}, {"segments", check_segments}, {"limits", check_limits},
        {"exponents", check_exponents}};
    for (const auto& g : groups)
        if (!strcmp(what, g.name)) return g.fn() ? 1 : 0;
    if (!strcmp(what, "check") || !strcmp(what, "all")) {
        fails += check_small();
        fails += check_lauum(512);
        fails += check_lauum(1152);
        fails += check_batched();
        printf("check: %s (%d failing groups)\n", fails ? "FAILED" : "ok", fails);
        fflush(stdout);
    }
    if ((!strcmp(what, "perf") || !strcmp(what, "all")) && fails == 0) {
        if (argc > 4) {
            perf(atoi(argv[2]), atoi(argv[3]), atoi(argv[4]), argc > 5 ? atoi(argv[5]) : 3);
        } else {
            perf(4096, 8, 0, 5);
            perf(8192, 12, 0, 5);
            perf(16384, 12, 0, 3);
            perf(16384, 24, 0, 3);
            perf(8192, 64, 1, 3);
            perf(16384, 128, 1, 2);
        }
    }
    return fails ? 1 : 0;
}
