// Development bench for the factorisation kernels (not part of the product library).
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -lineinfo -o tools/chol_lab tools/chol_lab.cu
//   ./tools/chol_lab [N ...]
// Times the leaf kernels (with clock64 phase stamps), DMMA GEMM shapes and the blocked / look-ahead
// Cholesky drivers on a Kac-Murdock-Szego test matrix, and cross-checks every variant against the first one.
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>

#include <vector>

#include "../gp-plus_b200/csrc/chol.cuh"

using namespace gpp;

#define CHECK(x)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (x);                                                                      \
        if (e_ != cudaSuccess) {                                                                   \
            fprintf(stderr, "%s:%d %s -> %s\n", __FILE__, __LINE__, #x, cudaGetErrorString(e_)); \
            exit(1);                                                                               \
        }                                                                                          \
    } while (0)

__global__ void fill_kms(double* A, long long ld, int n, double rho, double nug) {
    long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (long long)n * n) return;
    int i = (int)(idx / n), j = (int)(idx % n);
    double v = pow(rho, fabs((double)(i - j))) * (1.0 + 0.3 * cos(0.37 * i) * cos(0.37 * j));
    if (i == j) v += nug;
    A[(long long)i * ld + j] = v;
}

__global__ void maxdiff_lower(const double* A, const double* B, long long ld, int n, double* out) {
    long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    double d = 0.0;
    if (idx < (long long)n * n) {
        int i = (int)(idx / n), j = (int)(idx % n);
        if (j <= i) d = fabs(A[(long long)i * ld + j] - B[(long long)i * ld + j]);
    }
    for (int o = 16; o > 0; o >>= 1) d = fmax(d, __shfl_xor_sync(0xffffffffu, d, o));
    if ((threadIdx.x & 31) == 0 && d > 0.0) atomicMax((unsigned long long*)out, (unsigned long long)__double_as_longlong(d));
}

// residual of sampled entries: |(L L^T)_ij - A0_ij|
__global__ void resid_sample(const double* L, const double* A0, long long ld, int n, int ns, double* out) {
    int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= ns) return;
    unsigned h = 2654435761u * (unsigned)(s + 1);
    int i = (int)(h % (unsigned)n);
    h = h * 1664525u + 1013904223u;
    int j = (int)(h % (unsigned)(i + 1));
    double acc = 0.0;
    for (int k = 0; k <= j; k++) acc = fma(L[(long long)i * ld + k], L[(long long)j * ld + k], acc);
    double d = fabs(acc - A0[(long long)i * ld + j]);
    atomicMax((unsigned long long*)out, (unsigned long long)__double_as_longlong(d));
}

// |M_kk L_kk - I| on the diagonal 128-blocks, sampled rows
__global__ void inv_check(const double* L, const double* M, long long ld, int T, double* out) {
    int kb = blockIdx.x;
    int i = threadIdx.x;  // 128 threads: row i of the block, column = (i*7) % 128 and i
    const double* Lb = L + (long long)kb * 128 * ld + (long long)kb * 128;
    const double* Mb = M + (long long)kb * 128 * ld + (long long)kb * 128;
    for (int rep = 0; rep < 2; rep++) {
        int c = rep == 0 ? i : (i * 7) % 128;
        double acc = 0.0;
        for (int k = c; k <= i; k++) acc = fma(Mb[(long long)i * ld + k], Lb[(long long)k * ld + c], acc);
        double d = fabs(acc - (c == i ? 1.0 : 0.0));
        if (c > i) d = fabs(Mb[(long long)i * ld + c]);
        atomicMax((unsigned long long*)out, (unsigned long long)__double_as_longlong(d));
    }
}

static double read_max(double* d) {
    double h;
    CHECK(cudaMemcpy(&h, d, 8, cudaMemcpyDeviceToHost));
    CHECK(cudaMemset(d, 0, 8));
    return h;
}

struct Timer {
    cudaEvent_t a, b;
    Timer() { cudaEventCreate(&a); cudaEventCreate(&b); }
    void start(cudaStream_t s) { cudaEventRecord(a, s); }
    float stop(cudaStream_t s) {
        cudaEventRecord(b, s);
        cudaEventSynchronize(b);
        float ms;
        cudaEventElapsedTime(&ms, a, b);
        return ms;
    }
};


// ---- instruction latency probes (one warp, dependent chains) ------------------------------------
__global__ void lat_kernel(double* out, long long* cyc, double seed) {
    __shared__ double sh[64];
    const int lane = threadIdx.x;
    double x = seed + lane * 1e-3, y = 1.0 + seed;
    long long t0, t1;
    // dependent DFMA chain
    t0 = clock64();
#pragma unroll
    for (int i = 0; i < 64; i++) x = fma(x, y, 1e-9);
    t1 = clock64();
    if (lane == 0) cyc[0] = (t1 - t0) / 64;
    // dependent rsqrt chain
    double z = 2.0 + x * 1e-300;
    t0 = clock64();
#pragma unroll
    for (int i = 0; i < 16; i++) z = rsqrt(z) + 1.5;
    t1 = clock64();
    if (lane == 0) cyc[1] = (t1 - t0) / 16;
    // dependent sqrt chain
    t0 = clock64();
#pragma unroll
    for (int i = 0; i < 16; i++) z = sqrt(z) + 1.5;
    t1 = clock64();
    if (lane == 0) cyc[2] = (t1 - t0) / 16;
    // dependent division chain
    t0 = clock64();
#pragma unroll
    for (int i = 0; i < 16; i++) z = 1.0 / z + 1.5;
    t1 = clock64();
    if (lane == 0) cyc[3] = (t1 - t0) / 16;
    // dependent double shuffle chain
    t0 = clock64();
#pragma unroll
    for (int i = 0; i < 32; i++) z = __shfl_sync(0xffffffffu, z, (i * 7) & 31);
    t1 = clock64();
    if (lane == 0) cyc[4] = (t1 - t0) / 32;
    // shared-memory round trip: STS, syncwarp, broadcast LDS
    t0 = clock64();
#pragma unroll
    for (int i = 0; i < 32; i++) {
        sh[lane] = z;
        __syncwarp();
        z = sh[(i * 5) & 31] + 1e-12;
        __syncwarp();
    }
    t1 = clock64();
    if (lane == 0) cyc[5] = (t1 - t0) / 32;
    // dependent DMMA chain (same accumulator)
    double c0 = 0.0, c1 = 0.0;
    t0 = clock64();
#pragma unroll
    for (int i = 0; i < 64; i++) dmma884(c0, c1, x, y);
    t1 = clock64();
    if (lane == 0) cyc[6] = (t1 - t0) / 64;
    // independent DMMAs (16 accumulators), issue rate of one warp
    double a0[16], a1[16];
#pragma unroll
    for (int k = 0; k < 16; k++) { a0[k] = 0.0; a1[k] = 0.0; }
    t0 = clock64();
#pragma unroll
    for (int i = 0; i < 8; i++)
#pragma unroll
        for (int k = 0; k < 16; k++) dmma884(a0[k], a1[k], x, y);
    t1 = clock64();
    if (lane == 0) cyc[7] = (t1 - t0) / 128;
    double acc = c0 + c1;
#pragma unroll
    for (int k = 0; k < 16; k++) acc += a0[k] + a1[k];
    // MUFU.RSQ64H-based fast reciprocal sqrt: raw approximation + 2 Newton steps
    double w = 3.0 + z * 1e-300;
    t0 = clock64();
#pragma unroll
    for (int i = 0; i < 16; i++) {
        double r;
        asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(w));
        double e = fma(-w * r, r, 1.0);
        r = fma(0.5 * r, e, r);
        e = fma(-w * r, r, 1.0);
        r = fma(0.5 * r, e, r);
        w = r + 2.5;
    }
    t1 = clock64();
    if (lane == 0) cyc[8] = (t1 - t0) / 16;
    out[lane] = x + z + acc + w;
}

static void lat_lab(cudaStream_t st) {
    double* out;
    long long* cyc;
    CHECK(cudaMalloc(&out, 32 * 8));
    CHECK(cudaMalloc(&cyc, 16 * 8));
    for (int rep = 0; rep < 2; rep++) lat_kernel<<<1, 32, 0, st>>>(out, cyc, 0.5);
    CHECK(cudaStreamSynchronize(st));
    long long h[16];
    CHECK(cudaMemcpy(h, cyc, sizeof(h), cudaMemcpyDeviceToHost));
    printf("latency (cycles): dfma %lld  rsqrt() %lld  sqrt() %lld  div %lld  shfl.f64 %lld  sts+lds roundtrip %lld  dmma dep %lld  "
           "dmma indep issue %lld  rsqrt.approx+2NR %lld\n", h[0], h[1], h[2], h[3], h[4], h[5], h[6], h[7], h[8]);
    cudaFree(out);
    cudaFree(cyc);
}

static void leaf_lab(cudaStream_t st) {
    const int ld = 128;
    double *A0, *A, *M, *ldp, *mx;
    int* info;
    long long* prof;
    CHECK(cudaMalloc(&A0, 128 * 128 * 8));
    CHECK(cudaMalloc(&A, 128 * 128 * 8));
    CHECK(cudaMalloc(&M, 128 * 128 * 8));
    CHECK(cudaMalloc(&ldp, 8 * 4));
    CHECK(cudaMalloc(&mx, 8));
    CHECK(cudaMemset(mx, 0, 8));
    CHECK(cudaMalloc(&info, 4));
    CHECK(cudaMemset(info, 0, 4));
    CHECK(cudaMalloc(&prof, 16 * 8));
    fill_kms<<<(128 * 128 + 255) / 256, 256, 0, st>>>(A0, ld, 128, 0.9, 0.1);
    Timer tm;
    std::vector<double> Lref(128 * 128, 0.0), Lh(128 * 128), Mh(128 * 128);
    {   // textbook Cholesky on the host as the reference factor
        CHECK(cudaStreamSynchronize(st));
        CHECK(cudaMemcpy(Lref.data(), A0, 128 * 128 * 8, cudaMemcpyDeviceToHost));
        for (int j = 0; j < 128; j++) {
            double d = Lref[j * 128 + j];
            for (int k = 0; k < j; k++) d -= Lref[j * 128 + k] * Lref[j * 128 + k];
            d = sqrt(d);
            Lref[j * 128 + j] = d;
            for (int i = j + 1; i < 128; i++) {
                double v = Lref[i * 128 + j];
                for (int k = 0; k < j; k++) v -= Lref[i * 128 + k] * Lref[j * 128 + k];
                Lref[i * 128 + j] = v / d;
            }
        }
    }
    double ldref = 0.0;
    for (int j = 0; j < 128; j++) ldref += log(Lref[j * 128 + j]);
    float best = 1e9f, sum = 0;
    for (int it = 0; it < 12; it++) {
        CHECK(cudaMemcpyAsync(A, A0, 128 * 128 * 8, cudaMemcpyDeviceToDevice, st));
        CHECK(cudaMemsetAsync(M, 0, 128 * 128 * 8, st));
        CHECK(cudaMemsetAsync(prof, 0, 16 * 8, st));
        tm.start(st);
        CHECK(launch_leaf(A, ld, 0, M, ldp, info, st, prof));
        float ms = tm.stop(st);
        if (it >= 2) { best = fminf(best, ms); sum += ms; }
    }
    CHECK(cudaStreamSynchronize(st));
    int hinfo;
    double hld;
    CHECK(cudaMemcpy(&hinfo, info, 4, cudaMemcpyDeviceToHost));
    CHECK(cudaMemcpy(&hld, ldp, 8, cudaMemcpyDeviceToHost));
    CHECK(cudaMemcpy(Lh.data(), A, 128 * 128 * 8, cudaMemcpyDeviceToHost));
    CHECK(cudaMemcpy(Mh.data(), M, 128 * 128 * 8, cudaMemcpyDeviceToHost));
    inv_check<<<1, 128, 0, st>>>(A, M, ld, 1, mx);
    CHECK(cudaStreamSynchronize(st));
    double invres = read_max(mx);
    double dl = 0, du = 0;
    for (int i = 0; i < 128; i++)
        for (int j = 0; j < 128; j++) {
            if (j <= i) dl = fmax(dl, fabs(Lh[i * 128 + j] - Lref[i * 128 + j]));
            else du = fmax(du, fabs(Mh[i * 128 + j]));
        }
    printf("leaf: best %.1f us  avg %.1f us  info %d  |L - host chol|max %.3e  dlogdet %.3e  |M L - I|max %.3e  "
           "|M upper|max %.3e\n", best * 1e3, sum / 10 * 1e3, hinfo, dl, hld - ldref, invres, du);
    long long hp[16];
    CHECK(cudaMemcpy(hp, prof, sizeof(hp), cudaMemcpyDeviceToHost));
    const char* names[16] = {"start", "loaded", "potrf0", "trsm0", "syrk0", "potrf1", "trsm1", "syrk1", "potrf2",
                             "trsm2", "syrk2", "potrf3", "asm_done", "stored", "fact_done", "inv_warp_done"};
    printf("   stamps (cycles since start):");
    for (int i = 1; i < 16; i++) printf(" %s=%lld", names[i], hp[i] - hp[0]);
    printf("\n");
    cudaFree(A0); cudaFree(A); cudaFree(M); cudaFree(ldp); cudaFree(mx); cudaFree(info); cudaFree(prof);
}

static void gemm_lab(cudaStream_t st) {
    const int n = 8192;
    double *A, *B, *C;
    CHECK(cudaMalloc(&A, (size_t)n * n * 8));
    CHECK(cudaMalloc(&B, (size_t)n * n * 8));
    CHECK(cudaMalloc(&C, (size_t)n * n * 8));
    fill_kms<<<(int)(((long long)n * n + 255) / 256), 256, 0, st>>>(A, n, n, 0.99, 0.0);
    fill_kms<<<(int)(((long long)n * n + 255) / 256), 256, 0, st>>>(B, n, n, 0.98, 0.0);
    Timer tm;
    // full GEMM 8192^3
    GemmOp op = gemm_default();
    op.A = A; op.lda = n; op.B = B; op.ldb = n; op.C = C; op.ldc = n;
    op.tiles_m = op.tiles_m_last = n / 128; op.tiles_n = n / 128; op.khi_c = n / 128;
    for (int kc = 0; kc < 2; kc++) {
        bool akc = kc == 0, bkc = kc == 0;
        CHECK(launch_gemm(op, akc, bkc, 1, st));
        tm.start(st);
        for (int i = 0; i < 3; i++) CHECK(launch_gemm(op, akc, bkc, 1, st));
        float ms = tm.stop(st) / 3;
        printf("gemm layout=%s 8192^3: %.3f ms  %.2f TFLOP/s\n", kc == 0 ? "kc,kc" : "ks,ks", ms,
               2.0 * n * (double)n * n / (ms * 1e-3) / 1e12);
    }
    // SYRK-shaped trailing update: 60x60 lower tiles, K = 512
    for (int kblocks : {2, 4, 8}) {
        GemmOp s = gemm_default();
        s.A = A; s.lda = n; s.B = A; s.ldb = n; s.C = C; s.ldc = n;
        s.map = MAP_TRI; s.tiles_m = s.tiles_m_last = 60; s.tiles_n = 60; s.khi_c = kblocks; s.alpha = -1.0; s.beta = 1.0;
        CHECK(launch_gemm(s, true, true, 1, st));
        tm.start(st);
        for (int i = 0; i < 5; i++) CHECK(launch_gemm(s, true, true, 1, st));
        float ms = tm.stop(st) / 5;
        double fl = 60.0 * 61.0 / 2 * 2.0 * 128 * 128 * 128 * kblocks;
        printf("syrk 60x60 tri tiles K=%d: %.3f ms  %.2f TFLOP/s\n", kblocks * 128, ms, fl / (ms * 1e-3) / 1e12);
    }
    // TRSM-shaped: 100 x 1 tiles, K = 128; panel update: 100 x 3 tiles K = 128
    for (int tn : {1, 3}) {
        GemmOp s = gemm_default();
        s.A = A; s.lda = n; s.B = B; s.ldb = n; s.C = C; s.ldc = n;
        s.tiles_m = s.tiles_m_last = 60; s.tiles_n = tn; s.khi_c = 1;
        CHECK(launch_gemm(s, true, true, 1, st));
        tm.start(st);
        for (int i = 0; i < 10; i++) CHECK(launch_gemm(s, true, true, 1, st));
        float ms = tm.stop(st) / 10;
        printf("small 60x%d tiles K=128: %.1f us per launch (back to back)\n", tn, ms * 1e3);
    }
    cudaFree(A); cudaFree(B); cudaFree(C);
}

static void potrf_lab(int n, cudaStream_t st) {
    const int T = (n + 127) / 128;
    const long long ld = (long long)T * 128;
    double *A0, *A, *M, *Lref, *ldp, *mx;
    int* info;
    CHECK(cudaMalloc(&A0, (size_t)ld * ld * 8));
    CHECK(cudaMalloc(&A, (size_t)ld * ld * 8));
    CHECK(cudaMalloc(&M, (size_t)ld * ld * 8));
    CHECK(cudaMalloc(&Lref, (size_t)ld * ld * 8));
    CHECK(cudaMalloc(&ldp, 8 * T));
    CHECK(cudaMalloc(&mx, 8));
    CHECK(cudaMemset(mx, 0, 8));
    CHECK(cudaMalloc(&info, 4));
    CHECK(cudaMemset(info, 0, 4));
    CHECK(cudaMemset(M, 0, (size_t)ld * ld * 8));
    fill_kms<<<(int)((ld * ld + 255) / 256), 256, 0, st>>>(A0, ld, (int)ld, 0.999, 0.05);
    CholLookahead la;
    CHECK(la.init(T));
    Timer tm;
    struct Var { const char* name; int look, pb; };
    const Var vars[] = {{"blocked   P4", 0, 4}, {"lookahead P8", 1, 8}, {"lookahead P4", 1, 4}};
    const int nvars = (int)(sizeof(vars) / sizeof(vars[0]));
    const int nblk = (int)((ld * ld + 255) / 256);
    for (int v = 0; v < nvars; v++) {
        la.sched.panel_blocks = vars[v].pb;
        float best = 1e9f;
        for (int it = 0; it < 3; it++) {
            CHECK(cudaMemcpyAsync(A, A0, (size_t)ld * ld * 8, cudaMemcpyDeviceToDevice, st));
            tm.start(st);
            if (vars[v].look) CHECK(potrf_lookahead(A, M, (int)ld, T, ldp, info, st, la));
            else CHECK(potrf_blocked(A, M, (int)ld, T, ldp, info, st));
            best = fminf(best, tm.stop(st));
        }
        CHECK(cudaStreamSynchronize(st));
        int hinfo;
        CHECK(cudaMemcpy(&hinfo, info, 4, cudaMemcpyDeviceToHost));
        std::vector<double> hl(T);
        CHECK(cudaMemcpy(hl.data(), ldp, 8 * T, cudaMemcpyDeviceToHost));
        double logdet = 0;
        for (double x : hl) logdet += x;
        resid_sample<<<16, 256, 0, st>>>(A, A0, ld, (int)ld, 4096, mx);
        CHECK(cudaStreamSynchronize(st));
        double res = read_max(mx);
        inv_check<<<T, 128, 0, st>>>(A, M, ld, T, mx);
        CHECK(cudaStreamSynchronize(st));
        double invres = read_max(mx);
        double dl = -1;
        if (v == 0) CHECK(cudaMemcpy(Lref, A, (size_t)ld * ld * 8, cudaMemcpyDeviceToDevice));
        else {
            maxdiff_lower<<<nblk, 256, 0, st>>>(A, Lref, ld, (int)ld, mx);
            CHECK(cudaStreamSynchronize(st));
            dl = read_max(mx);
        }
        printf("potrf N=%d %s: %.3f ms  %.2f TFLOP/s  info %d  sum log L_jj %.12g  resid %.2e  |ML-I| %.2e  |dL| vs v0 %.2e\n",
               n, vars[v].name, best, (double)n * n * n / 3.0 / (best * 1e-3) / 1e12, hinfo, logdet, res, invres, dl);
        fflush(stdout);
    }
    la.destroy();
    cudaFree(A0); cudaFree(A); cudaFree(M); cudaFree(Lref); cudaFree(ldp); cudaFree(mx); cudaFree(info);
}

int main(int argc, char** argv) {
    CHECK(cudaSetDevice(0));
    CHECK(chol_set_attributes());
    cudaStream_t st;
    CHECK(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
    lat_lab(st);
    leaf_lab(st);
    if (getenv("LAB_GEMM")) gemm_lab(st);
    std::vector<int> ns;
    for (int i = 1; i < argc; i++) ns.push_back(atoi(argv[i]));
    if (ns.empty()) ns = {2048, 8192, 16384};
    for (int n : ns) potrf_lab(n, st);
    return 0;
}
