// pairdist.cuh -- the FP64 squared-distance tile of spatial.cu's distance pass (K14), as modal.cu (K15) uses it.
// spatial.cu keeps its own copy: calling this helper from spatial_dist_kernel renumbers the PTX registers of the
// accumulator and changes that kernel's register allocation (DESIGN K15).
//
// A block of SP_THREADS = 16 x 16 threads computes d2[q][s] = sum_f (x_q,f - x_s,f)^2 for SP_BQ = 64 query rows and
// SP_BS = 128 sample rows, streaming f through shared memory in double-buffered cp.async chunks of SP_BK.  Thread
// (tx, ty) holds the register micro-tile acc[i][j] of query q0 + ty + 16 i and sample s0 + tx + 16 j.  Each d2 is
// accumulated in f order with __dsub_rn / __fma_rn alone, so it depends on the two rows and nothing else: d2(a, b) and
// d2(b, a) are equal bit for bit ((a - b)^2 = (b - a)^2 in IEEE arithmetic), and d2(a, a) = +0.
#pragma once

#include "common.cuh"

namespace sd {

constexpr int SP_THREADS = 256;      // 16 x 16 threads
constexpr int SP_TQ = 4;             // register micro-tile: queries ...
constexpr int SP_TS = 8;             // ... x samples (distance pass) or x features (sum pass), strided by 16
constexpr int SP_BQ = 16 * SP_TQ;    // 64 queries per block
constexpr int SP_BS = 16 * SP_TS;    // 128 samples / features per block
constexpr int SP_BK = 16;            // reduction chunk staged in shared memory

__device__ __forceinline__ void cp_async8(double *dst, const double *src, bool valid) {
    const unsigned s = (unsigned)__cvta_generic_to_shared(dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;\n" ::"r"(s), "l"(src), "r"(valid ? 8 : 0));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
__device__ __forceinline__ void cp_async_wait1() { asm volatile("cp.async.wait_group 1;\n" ::); }

// rows [r0, r0 + R) x columns [c0, c0 + SP_BK) of a row-major matrix (row r at base + idx(r) * ld) into dst[k][r ^ k]:
// transposed, XOR-swizzled so that the 16 columns a half-warp copies land in distinct banks; out of range -> 0
template <int R>
__device__ __forceinline__ void stage_t(double (*dst)[R], const double *__restrict__ base, const i64 *__restrict__ idx,
                                        i64 r0, i64 nrows, i64 ld, i64 c0, i64 ncols) {
#pragma unroll
    for (int e = threadIdx.x; e < R * SP_BK; e += SP_THREADS) {
        const int r = e / SP_BK, k = e % SP_BK;
        const i64 gr = r0 + r, gc = c0 + k;
        const bool ok = gr < nrows && gc < ncols;
        cp_async8(&dst[k][r ^ k], ok ? base + (idx ? idx[gr] : gr) * ld + gc : base, ok);
    }
}

// rows [r0, r0 + SP_BK) x columns [c0, c0 + C) into dst[k][c] (as stored); out of range -> 0
template <int C>
__device__ __forceinline__ void stage_n(double (*dst)[C], const double *__restrict__ base, i64 r0, i64 nrows, i64 ld,
                                        i64 c0, i64 ncols) {
#pragma unroll
    for (int e = threadIdx.x; e < C * SP_BK; e += SP_THREADS) {
        const int k = e / C, c = e % C;
        const i64 gr = r0 + k, gc = c0 + c;
        const bool ok = gr < nrows && gc < ncols;
        cp_async8(&dst[k][c], ok ? base + gr * ld + gc : base, ok);
    }
}

// acc[i][j] += d2 of query row Q[idx(q0 + ty + 16 i) * F] (idx = qidx or the identity; rows >= nq read as 0) and
// sample row S[(s0 + tx + 16 j) * F] (rows >= nS read as 0); the caller zeroes acc.  Ends with a __syncthreads, so the
// caller may reuse As and Bs.
__device__ __forceinline__ void sq_dist_tile(double (*As)[SP_BK][SP_BQ], double (*Bs)[SP_BK][SP_BS], const int tx,
                                             const int ty, const double *__restrict__ Q, const i64 *__restrict__ qidx,
                                             const i64 q0, const i64 nq, const double *__restrict__ S, const i64 s0,
                                             const i64 nS, const i64 F, double (&acc)[SP_TQ][SP_TS]) {
    const i64 nk = ceil_div(F, SP_BK);
    stage_t<SP_BQ>(As[0], Q, qidx, q0, nq, F, 0, F);
    stage_t<SP_BS>(Bs[0], S, nullptr, s0, nS, F, 0, F);
    cp_async_commit();
    for (i64 kc = 0; kc < nk; ++kc) {
        const int b = (int)(kc & 1);
        if (kc + 1 < nk) {
            stage_t<SP_BQ>(As[b ^ 1], Q, qidx, q0, nq, F, (kc + 1) * SP_BK, F);
            stage_t<SP_BS>(Bs[b ^ 1], S, nullptr, s0, nS, F, (kc + 1) * SP_BK, F);
        }
        cp_async_commit();
        cp_async_wait1();
        __syncthreads();
#pragma unroll
        for (int k = 0; k < SP_BK; ++k) {
            double a[SP_TQ], s[SP_TS];
#pragma unroll
            for (int i = 0; i < SP_TQ; ++i) a[i] = As[b][k][(ty + 16 * i) ^ k];
#pragma unroll
            for (int j = 0; j < SP_TS; ++j) s[j] = Bs[b][k][(tx + 16 * j) ^ k];
#pragma unroll
            for (int i = 0; i < SP_TQ; ++i)
#pragma unroll
                for (int j = 0; j < SP_TS; ++j) {
                    const double d = __dsub_rn(a[i], s[j]);
                    acc[i][j] = __fma_rn(d, d, acc[i][j]);
                }
        }
        __syncthreads();
    }
}

}  // namespace sd
