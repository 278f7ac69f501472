// FP64 operand -> 7 signed base-256 digit planes (int8) + one power-of-two scale per operand row, for oz_gemm.cuh.
//
//   x[r,k] = scale[r] * sum_{p<7} d_p[r,k] 256^-(p+1)  + t,   0 <= t < scale[r] 2^-56,   d_p in [-128, 127], |d_0| <= 64
//
// scale[r] = 2^(e+2) with 2^(e-1) <= max_k |x[r,k]| < 2^e, so |x| / scale < 1/4 and v = floor(x / scale * 2^56) is an
// exact 55-bit integer; its balanced base-256 digits come out of integer arithmetic, least significant first
// (d = sign-extended low byte, v = (v - d) >> 8).  Planes are stored [plane][row][k] with k contiguous ("K-major"):
//   split_rows : operand given as [row][k]  (k contiguous in memory)  -> coalesced both ways
//   split_cols : operand given as [k][row]  (row contiguous)          -> transposed through shared memory
// Every kernel takes already-offset pointers; rows / k extents are multiples of 64.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "oz_gemm.cuh"

namespace gpp {

__device__ __forceinline__ double oz_scale_from_max(double amax, double2& inv56) {
    // amax = m 2^ex (m in [0.5,1)): scale = 2^(ex+2); x * 2^56 / scale = (x * inv56.x) * inv56.y with
    // inv56.x * inv56.y = 2^(54-ex).  That power of two overflows a double for rows with a maximum below 2^-970, so it
    // is applied as two exact multiplications there (inv56.y = 2^512); for every other row inv56.y = 1.
    // Zero rows: scale 1, digits 0.
    if (!(amax > 0.0) || !(amax < 1.0e300)) {  // zero, NaN or infinite rows: keep them finite, the caller's status flags the NaN
        inv56 = make_double2(0.0, 0.0);
        return 1.0;
    }
    int ex;
    frexp(amax, &ex);
    const int e56 = 56 - (ex + 2);
    inv56 = e56 <= 1023 ? make_double2(ldexp(1.0, e56), 1.0) : make_double2(ldexp(1.0, e56 - 512), ldexp(1.0, 512));
    return ldexp(1.0, ex + 2);
}

__device__ __forceinline__ void oz_digits(double x, double2 inv56, int8_t (&d)[OZ_S]) {
    long long v = __double2ll_rd((x * inv56.x) * inv56.y);
#pragma unroll
    for (int p = OZ_S - 1; p >= 0; p--) {
        const long long lo = (long long)(int8_t)(v & 0xff);
        d[p] = (int8_t)lo;
        v = (v - lo) >> 8;
    }
}

// ---- k-contiguous operand ----------------------------------------------------------------------------------
// One warp per row: pass 1 row maximum, pass 2 digits (the row comes back from L1/L2).  kcols % 16 == 0.
// batched: blockIdx.y = batch entry; element (r,k) of entry z at X[z*x_zs + r*ld + k], plane element at
// planes[p*plane_stride + z*pl_zs + r*pitch + k], scale[z*sc_zs + r].
__global__ void __launch_bounds__(256) oz_split_rows_kernel(const double* __restrict__ X, long long ld, long long x_zs,
                                                            int rows, int rows_last, int kcols_all, int kcols_last,
                                                            int8_t* __restrict__ planes,
                                                            long long pitch, long long plane_stride, long long pl_zs,
                                                            double* __restrict__ scale, long long sc_zs) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int z = blockIdx.y;
    const int nrows = (z == (int)gridDim.y - 1) ? rows_last : rows;
    const int kcols = (z == (int)gridDim.y - 1) ? kcols_last : kcols_all;
    const int r = blockIdx.x * 8 + warp;
    if (r >= nrows) return;
    const double* x = X + (long long)z * x_zs + (long long)r * ld;
    double amax = 0.0;
    for (int k = lane * 2; k < kcols; k += 64) {
        const double2 v = *reinterpret_cast<const double2*>(x + k);
        amax = fmax(amax, fmax(fabs(v.x), fabs(v.y)));
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) amax = fmax(amax, __shfl_xor_sync(0xffffffffu, amax, o));
    double2 inv56;
    const double sc = oz_scale_from_max(amax, inv56);
    if (lane == 0) scale[(long long)z * sc_zs + r] = sc;
    int8_t* out = planes + (long long)z * pl_zs + (long long)r * pitch;
    for (int k0 = lane * 16; k0 < kcols; k0 += 512) {
        int8_t dg[OZ_S][16];
#pragma unroll
        for (int e = 0; e < 16; e += 2) {
            const double2 v = *reinterpret_cast<const double2*>(x + k0 + e);
            int8_t d0[OZ_S], d1[OZ_S];
            oz_digits(v.x, inv56, d0);
            oz_digits(v.y, inv56, d1);
#pragma unroll
            for (int p = 0; p < OZ_S; p++) { dg[p][e] = d0[p]; dg[p][e + 1] = d1[p]; }
        }
#pragma unroll
        for (int p = 0; p < OZ_S; p++) {
            int4 w;
            w.x = (int)((uint32_t)(uint8_t)dg[p][0] | ((uint32_t)(uint8_t)dg[p][1] << 8) | ((uint32_t)(uint8_t)dg[p][2] << 16) | ((uint32_t)(uint8_t)dg[p][3] << 24));
            w.y = (int)((uint32_t)(uint8_t)dg[p][4] | ((uint32_t)(uint8_t)dg[p][5] << 8) | ((uint32_t)(uint8_t)dg[p][6] << 16) | ((uint32_t)(uint8_t)dg[p][7] << 24));
            w.z = (int)((uint32_t)(uint8_t)dg[p][8] | ((uint32_t)(uint8_t)dg[p][9] << 8) | ((uint32_t)(uint8_t)dg[p][10] << 16) | ((uint32_t)(uint8_t)dg[p][11] << 24));
            w.w = (int)((uint32_t)(uint8_t)dg[p][12] | ((uint32_t)(uint8_t)dg[p][13] << 8) | ((uint32_t)(uint8_t)dg[p][14] << 16) | ((uint32_t)(uint8_t)dg[p][15] << 24));
            *reinterpret_cast<int4*>(out + (long long)p * plane_stride + k0) = w;
        }
    }
}

// ---- row-contiguous operand (transposed planes) -------------------------------------------------------------
// pass 1: colmax[c] = max_k |X[k][c]| as the bit pattern of a non-negative double (atomicMax on 64-bit integers);
// colmax must be zeroed first.  lower != 0: only k >= (c / 128) * 128 is visited (lower-triangular tile storage).
__global__ void __launch_bounds__(256) oz_colmax_kernel(const double* __restrict__ X, long long ld, long long x_zs, int krows,
                                                        int krows_last, int cols, int lower, unsigned long long* colmax,
                                                        long long cm_zs) {
    const int z = blockIdx.z;
    const int nk = (z == (int)gridDim.z - 1) ? krows_last : krows;
    const int c = blockIdx.x * 256 + threadIdx.x;
    const int kchunk = blockIdx.y * 128;
    if (c >= cols || kchunk >= nk) return;
    if (lower && kchunk < (c / 128) * 128) return;
    const double* x = X + (long long)z * x_zs + (long long)kchunk * ld + c;
    double amax = 0.0;
    const int kend = (nk - kchunk < 128) ? (nk - kchunk) : 128;
#pragma unroll 8
    for (int k = 0; k < kend; k++) amax = fmax(amax, fabs(x[(long long)k * ld]));
    if (amax > 0.0) atomicMax(colmax + (long long)z * cm_zs + c, (unsigned long long)__double_as_longlong(amax));
    else if (amax != amax) atomicMax(colmax + (long long)z * cm_zs + c, 0x7ff8000000000000ull);
}

// pass 2: one CTA per 64(k) x 64(c) tile; digits staged as [plane][c][k] bytes in shared memory, written out in
// 16-byte pieces along k.  Also writes scale[c] (by the CTAs of the first visited k tile of every column block).
constexpr int OZ_TP = 64 + 16;  // shared row pitch in bytes (16-byte aligned rows, conflict-light)
__global__ void __launch_bounds__(256) oz_split_cols_kernel(const double* __restrict__ X, long long ld, long long x_zs,
                                                            int krows, int krows_last, int cols, int lower,
                                                            const unsigned long long* __restrict__ colmax, long long cm_zs,
                                                            int8_t* __restrict__ planes, long long pitch,
                                                            long long plane_stride, long long pl_zs,
                                                            double* __restrict__ scale, long long sc_zs) {
    __shared__ __align__(16) int8_t sm[OZ_S][64][OZ_TP];
    __shared__ double2 s_inv[64];
    const int z = blockIdx.z;
    const int nk = (z == (int)gridDim.z - 1) ? krows_last : krows;
    const int c0 = blockIdx.x * 64, k0 = blockIdx.y * 64;
    if (k0 >= nk) return;
    if (lower && k0 < (c0 / 128) * 128) return;
    const int tid = threadIdx.x;
    if (tid < 64) {
        const double amax = __longlong_as_double((long long)colmax[(long long)z * cm_zs + c0 + tid]);
        double2 inv56;
        const double sc = oz_scale_from_max(amax, inv56);
        s_inv[tid] = inv56;
        const int kfirst = lower ? (c0 / 128) * 128 : 0;
        if (k0 == kfirst) scale[(long long)z * sc_zs + c0 + tid] = sc;
    }
    __syncthreads();
    const double* x = X + (long long)z * x_zs + (long long)k0 * ld + c0;
    // thread -> column pair (2 * (tid & 31)), eight consecutive k rows 8 * (tid >> 5) + i: one 8-byte store per
    // (plane, column) instead of eight byte stores
    const int cp = (tid & 31) * 2;
    const int kb = (tid >> 5) * 8;
    const double2 i0 = s_inv[cp], i1 = s_inv[cp + 1];
    unsigned long long w0[OZ_S], w1[OZ_S];
#pragma unroll
    for (int p = 0; p < OZ_S; p++) { w0[p] = 0ull; w1[p] = 0ull; }
#pragma unroll
    for (int i = 0; i < 8; i++) {
        const double2 v = *reinterpret_cast<const double2*>(x + (long long)(kb + i) * ld + cp);
        int8_t d0[OZ_S], d1[OZ_S];
        oz_digits(v.x, i0, d0);
        oz_digits(v.y, i1, d1);
#pragma unroll
        for (int p = 0; p < OZ_S; p++) {
            w0[p] |= (unsigned long long)(uint8_t)d0[p] << (8 * i);
            w1[p] |= (unsigned long long)(uint8_t)d1[p] << (8 * i);
        }
    }
#pragma unroll
    for (int p = 0; p < OZ_S; p++) {
        *reinterpret_cast<unsigned long long*>(&sm[p][cp][kb]) = w0[p];
        *reinterpret_cast<unsigned long long*>(&sm[p][cp + 1][kb]) = w1[p];
    }
    __syncthreads();
    int8_t* out = planes + (long long)z * pl_zs + (long long)c0 * pitch + k0;
    // 7 planes x 64 columns x 4 pieces of 16 bytes
    for (int idx = tid; idx < OZ_S * 64 * 4; idx += 256) {
        const int p = idx >> 8, rem = idx & 255, c = rem >> 2, piece = rem & 3;
        const int4 w = *reinterpret_cast<const int4*>(&sm[p][c][piece * 16]);
        *reinterpret_cast<int4*>(out + (long long)p * plane_stride + (long long)c * pitch + piece * 16) = w;
    }
}

// ---- launchers ----------------------------------------------------------------------------------------------
struct OzPlanes {
    int8_t* planes = nullptr;     // [OZ_S][rows][pitch]
    double* scale = nullptr;      // [rows]
    unsigned long long* colmax = nullptr;  // [rows] scratch of split_cols
    long long rows = 0, pitch = 0;
    long long plane_stride() const { return rows * pitch; }
};

// rows x kcols block of a k-contiguous operand; destination plane coordinates (row_dst, k_dst)
inline cudaError_t oz_split_rows(const double* X, long long ld, long long x_zs, int rows, int rows_last, int kcols,
                                 const OzPlanes& P, long long row_dst, long long k_dst, long long dst_zs_row,
                                 long long dst_zs_k, int nbatch, cudaStream_t st, int kcols_last = -1) {
    if (rows <= 0 || kcols <= 0 || nbatch <= 0) return cudaSuccess;
    count_launch();
    dim3 grid((rows + 7) / 8, nbatch);
    oz_split_rows_kernel<<<grid, 256, 0, st>>>(X, ld, x_zs, rows, rows_last, kcols, kcols_last < 0 ? kcols : kcols_last,
                                               P.planes + row_dst * P.pitch + k_dst,
                                               P.pitch, P.plane_stride(), dst_zs_row * P.pitch + dst_zs_k, P.scale + row_dst,
                                               dst_zs_row);
    return cudaGetLastError();
}

// krows x cols block of a row-contiguous operand X[k][c]; destination plane coordinates (row_dst = c, k_dst)
inline cudaError_t oz_split_cols(const double* X, long long ld, long long x_zs, int krows, int krows_last, int cols, int lower,
                                 const OzPlanes& P, long long row_dst, long long k_dst, long long dst_zs_row,
                                 long long dst_zs_k, int nbatch, cudaStream_t st) {
    if (krows <= 0 || cols <= 0 || nbatch <= 0) return cudaSuccess;
    // column maxima of every batch entry (entries own disjoint plane rows)
    for (int zb = 0; zb < nbatch; zb++) {
        cudaError_t e = cudaMemsetAsync(P.colmax + row_dst + zb * dst_zs_row, 0, sizeof(unsigned long long) * cols, st);
        if (e != cudaSuccess) return e;
    }
    count_launch(2);
    dim3 g1((cols + 255) / 256, (krows + 127) / 128, nbatch);
    oz_colmax_kernel<<<g1, 256, 0, st>>>(X, ld, x_zs, krows, krows_last, cols, lower, P.colmax + row_dst, dst_zs_row);
    dim3 g2(cols / 64, (krows + 63) / 64, nbatch);
    oz_split_cols_kernel<<<g2, 256, 0, st>>>(X, ld, x_zs, krows, krows_last, cols, lower, P.colmax + row_dst, dst_zs_row,
                                             P.planes + row_dst * P.pitch + k_dst, P.pitch, P.plane_stride(),
                                             dst_zs_row * P.pitch + dst_zs_k, P.scale + row_dst, dst_zs_row);
    return cudaGetLastError();
}

}  // namespace gpp
