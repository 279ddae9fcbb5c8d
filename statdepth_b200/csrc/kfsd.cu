// kfsd.cu -- kernelized functional spatial depth (K16): spatial depth after the Gaussian feature map phi of the kernel
// k(x, y) = exp(c ||x - y||^2), c = -1 / sigma^2.  A curve is the vector of its F = T d values.  With
//   e(x, y) = 1 - k(x, y) = -expm1(c d2(x, y)),   w_qj = 1 / sqrt(2 e_qj) for e_qj > 0, else 0,
// the squared norm of the sum of the feature-space unit vectors (phi(x_q) - phi(x_j)) / ||.|| over the sample is
//   r_q^2 = 2 A_q B_q - Q_q,   A_q = sum_j w_qj,   B_q = sum_j w_qj e_qj,   Q_q = w_q^T E w_q,
// E [nS][nS] the sample's matrix of e_ij, and depth = 1 - r_q / n_pop (formed by the host).
//
// Four kernels on the FP64 pipe (tcgen05.mma has no f64 kind), the first two on pairdist.cuh's d2 tile:
//   gram pass     E[i][j] = -expm1(c d2(x_i, x_j)) over (64 x 128) tiles; d2(a, b) == d2(b, a) bit for bit, so E is
//                 symmetric bit for bit, and E[i][i] = 0.  A d2 that overflows sets ST_OVERFLOW.
//   weight pass   grid (sample tiles x query tiles): one row block of W[q][s] = w_qs, and one partial (sum w, sum w e)
//                 per (query, sample tile).
//   quad pass     a 64-query x 128-column tile of Z = W E, the sample index k streamed through double-buffered
//                 cp.async shared chunks in k order; its epilogue dots each row of Z with w_q over the tile's columns
//                 and writes one partial per (query, column tile).
//   finish        adds a query's partials in tile order and forms r = sqrt(max(2 A B - Q, 0)) in one expression.
// No float atomics and no split of k: a query's bits depend on its row, the sample and the tile sizes alone, not on
// the other queries, the row block or the rank.  Out of sample, the pooled in-sample call of S + [g] differs only by
// g's own column, whose weight is 0: every term it adds is an exact +0, so both calls give the same bits.
#include <float.h>

#include "pairdist.cuh"

namespace sd {

constexpr size_t KF_W_BUDGET = 1ull << 30;  // bytes of one W row block (BUF_KFSD)

// grid (ceil(n / SP_BS), ceil(n / SP_BQ)): E [n][n] of the rows X [n, F]
__global__ void __launch_bounds__(SP_THREADS) kfsd_gram_kernel(const double *__restrict__ X, const i64 n, const i64 F,
                                                               const double c, double *__restrict__ E,
                                                               int *__restrict__ status) {
    __shared__ __align__(16) double As[2][SP_BK][SP_BQ];
    __shared__ __align__(16) double Bs[2][SP_BK][SP_BS];
    const int tx = threadIdx.x % 16, ty = threadIdx.x / 16;
    const i64 q0 = (i64)blockIdx.y * SP_BQ, s0 = (i64)blockIdx.x * SP_BS;
    double acc[SP_TQ][SP_TS];
#pragma unroll
    for (int i = 0; i < SP_TQ; ++i)
#pragma unroll
        for (int j = 0; j < SP_TS; ++j) acc[i][j] = 0.0;
    sq_dist_tile(As, Bs, tx, ty, X, nullptr, q0, n, X, s0, n, F, acc);
    bool overflow = false;
#pragma unroll
    for (int i = 0; i < SP_TQ; ++i) {
        const i64 q = q0 + ty + 16 * i;
        if (q >= n) continue;
#pragma unroll
        for (int j = 0; j < SP_TS; ++j) {
            const i64 s = s0 + tx + 16 * j;
            if (s >= n) continue;
            const double d2 = acc[i][j];
            if (!(d2 <= DBL_MAX)) overflow = true;
            E[q * n + s] = -expm1(__dmul_rn(c, d2));
        }
    }
    if (overflow) atomicOr(status, ST_OVERFLOW);
}

// grid (ceil(nS / SP_BS), ceil(nq / SP_BQ)).  Queries: rows Q[idx(q) * F] (idx = qidx or q).  W [nq][nS];
// pa / pb [nq][gridDim.x]: sum_s w and sum_s w e over this tile's columns, each thread in column order, then a fixed
// butterfly over the 16 lanes of a row.
__global__ void __launch_bounds__(SP_THREADS) kfsd_weight_kernel(const double *__restrict__ Q,
                                                                 const i64 *__restrict__ qidx, const i64 nq,
                                                                 const double *__restrict__ S, const i64 nS,
                                                                 const i64 F, const double c, double *__restrict__ W,
                                                                 double *__restrict__ pa, double *__restrict__ pb,
                                                                 int *__restrict__ status) {
    __shared__ __align__(16) double As[2][SP_BK][SP_BQ];
    __shared__ __align__(16) double Bs[2][SP_BK][SP_BS];
    const int tx = threadIdx.x % 16, ty = threadIdx.x / 16;
    const i64 q0 = (i64)blockIdx.y * SP_BQ, s0 = (i64)blockIdx.x * SP_BS;
    double acc[SP_TQ][SP_TS];
#pragma unroll
    for (int i = 0; i < SP_TQ; ++i)
#pragma unroll
        for (int j = 0; j < SP_TS; ++j) acc[i][j] = 0.0;
    sq_dist_tile(As, Bs, tx, ty, Q, qidx, q0, nq, S, s0, nS, F, acc);
    bool overflow = false;
#pragma unroll
    for (int i = 0; i < SP_TQ; ++i) {
        const i64 q = q0 + ty + 16 * i;
        double a = 0.0, b = 0.0;
#pragma unroll
        for (int j = 0; j < SP_TS; ++j) {
            const i64 s = s0 + tx + 16 * j;
            if (q < nq && s < nS) {
                const double d2 = acc[i][j];
                if (!(d2 <= DBL_MAX)) overflow = true;
                const double e = -expm1(__dmul_rn(c, d2));
                const double w = e > 0.0 ? __drcp_rn(__dsqrt_rn(__dmul_rn(2.0, e))) : 0.0;
                W[q * nS + s] = w;
                a = __dadd_rn(a, w);
                b = __fma_rn(w, e, b);
            }
        }
#pragma unroll
        for (int m = 1; m < 16; m <<= 1) {
            a = __dadd_rn(a, __shfl_xor_sync(0xffffffffu, a, m));
            b = __dadd_rn(b, __shfl_xor_sync(0xffffffffu, b, m));
        }
        if (tx == 0 && q < nq) {
            pa[q * gridDim.x + blockIdx.x] = a;
            pb[q * gridDim.x + blockIdx.x] = b;
        }
    }
    if (overflow) atomicOr(status, ST_OVERFLOW);
}

// grid (ceil(nS / SP_BS), ceil(nq / SP_BQ)).  Z[q][j] = sum_k W[q][k] E[k][j] for this block's 64 queries and 128
// columns, k in order (one FMA chain per output); pq[q * gridDim.x + blockIdx.x] = sum over the block's columns j of
// Z[q][j] W[q][j] (each thread in column order, then the butterfly).
__global__ void __launch_bounds__(SP_THREADS) kfsd_quad_kernel(const double *__restrict__ W, const i64 nq,
                                                               const double *__restrict__ E, const i64 nS,
                                                               double *__restrict__ pq) {
    __shared__ __align__(16) double Ws[2][SP_BK][SP_BQ];
    __shared__ __align__(16) double Es[2][SP_BK][SP_BS];
    const int tx = threadIdx.x % 16, ty = threadIdx.x / 16;
    const i64 q0 = (i64)blockIdx.y * SP_BQ, j0 = (i64)blockIdx.x * SP_BS;
    double acc[SP_TQ][SP_TS];
#pragma unroll
    for (int i = 0; i < SP_TQ; ++i)
#pragma unroll
        for (int j = 0; j < SP_TS; ++j) acc[i][j] = 0.0;
    const i64 nk = ceil_div(nS, SP_BK);
    stage_t<SP_BQ>(Ws[0], W, nullptr, q0, nq, nS, 0, nS);
    stage_n<SP_BS>(Es[0], E, 0, nS, nS, j0, nS);
    cp_async_commit();
    for (i64 kc = 0; kc < nk; ++kc) {
        const int b = (int)(kc & 1);
        if (kc + 1 < nk) {
            stage_t<SP_BQ>(Ws[b ^ 1], W, nullptr, q0, nq, nS, (kc + 1) * SP_BK, nS);
            stage_n<SP_BS>(Es[b ^ 1], E, (kc + 1) * SP_BK, nS, nS, j0, nS);
        }
        cp_async_commit();
        cp_async_wait1();
        __syncthreads();
#pragma unroll
        for (int k = 0; k < SP_BK; ++k) {
            double w[SP_TQ], e[SP_TS];
#pragma unroll
            for (int i = 0; i < SP_TQ; ++i) w[i] = Ws[b][k][(ty + 16 * i) ^ k];
#pragma unroll
            for (int j = 0; j < SP_TS; ++j) e[j] = Es[b][k][tx + 16 * j];
#pragma unroll
            for (int i = 0; i < SP_TQ; ++i)
#pragma unroll
                for (int j = 0; j < SP_TS; ++j) acc[i][j] = __fma_rn(w[i], e[j], acc[i][j]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < SP_TQ; ++i) {
        const i64 q = q0 + ty + 16 * i;
        double v = 0.0;
#pragma unroll
        for (int j = 0; j < SP_TS; ++j) {
            const i64 s = j0 + tx + 16 * j;
            if (q < nq && s < nS) v = __fma_rn(acc[i][j], W[q * nS + s], v);
        }
#pragma unroll
        for (int m = 1; m < 16; m <<= 1) v = __dadd_rn(v, __shfl_xor_sync(0xffffffffu, v, m));
        if (tx == 0 && q < nq) pq[q * gridDim.x + blockIdx.x] = v;
    }
}

__global__ void kfsd_finish_kernel(const double *__restrict__ pa, const double *__restrict__ pb,
                                   const double *__restrict__ pq, const i64 nq, const i64 ntile,
                                   double *__restrict__ r) {
    const i64 q = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= nq) return;
    double a = 0.0, b = 0.0, z = 0.0;
    for (i64 t = 0; t < ntile; ++t) {
        a = __dadd_rn(a, pa[q * ntile + t]);
        b = __dadd_rn(b, pb[q * ntile + t]);
        z = __dadd_rn(z, pq[q * ntile + t]);
    }
    const double r2 = __fma_rn(__dmul_rn(2.0, a), b, -z);
    r[q] = __dsqrt_rn(r2 > 0.0 ? r2 : 0.0);
}

int kfsd_gram_device(sd_ctx *ctx, const double *dX, i64 n, i64 F, double c, double *dE) {
    kfsd_gram_kernel<<<dim3((unsigned)ceil_div(n, SP_BS), (unsigned)ceil_div(n, SP_BQ)), SP_THREADS, 0,
                       ctx->stream>>>(dX, n, F, c, dE, ctx->d_status);
    ctx->last.launches += 1;
    SD_CUDA(cudaGetLastError());
    return SD_OK;
}

// r of the nq queries (rows dQ[idx(q) * F], idx = d_qidx or q) against the sample rows dS [nS, F] with the sample's
// E [nS][nS] (dE; nullptr: built here, into BUF_KFSD).  Row blocks of queries keep W within KF_W_BUDGET; a query's
// bits do not depend on the row block.
int kfsd_device(sd_ctx *ctx, const double *dQ, const i64 *d_qidx, i64 nq, const double *dS, i64 nS, i64 F, double c,
                const double *dE, double *d_r) {
    if (nq == 0) return SD_OK;
    const i64 ntile = ceil_div(nS, SP_BS);
    i64 RB = (i64)(KF_W_BUDGET / ((size_t)nS * sizeof(double))) / SP_BQ * SP_BQ;
    if (RB < SP_BQ) RB = SP_BQ;
    if (RB > 65535ll * SP_BQ) RB = 65535ll * SP_BQ;  // grid.y
    if (RB > ceil_div(nq, SP_BQ) * SP_BQ) RB = ceil_div(nq, SP_BQ) * SP_BQ;
    const size_t nE = dE ? 0 : (size_t)nS * nS;
    SD_TRY(ctx->buf[BUF_KFSD].reserve((nE + (size_t)RB * (nS + 3 * ntile)) * sizeof(double)));
    double *base = ctx->buf[BUF_KFSD].as<double>();
    double *dW = base + nE;
    double *pa = dW + (size_t)RB * nS, *pb = pa + (size_t)RB * ntile, *pq = pb + (size_t)RB * ntile;
    if (!dE) {
        SD_TRY(kfsd_gram_device(ctx, dS, nS, F, c, base));
        dE = base;
    }
    cudaStream_t st = ctx->stream;
    for (i64 r0 = 0; r0 < nq; r0 += RB) {
        const i64 rows = nq - r0 < RB ? nq - r0 : RB;
        const double *Q = d_qidx ? dQ : dQ + r0 * F;
        const i64 *qi = d_qidx ? d_qidx + r0 : nullptr;
        const dim3 grid((unsigned)ntile, (unsigned)ceil_div(rows, SP_BQ));
        kfsd_weight_kernel<<<grid, SP_THREADS, 0, st>>>(Q, qi, rows, dS, nS, F, c, dW, pa, pb, ctx->d_status);
        kfsd_quad_kernel<<<grid, SP_THREADS, 0, st>>>(dW, rows, dE, nS, pq);
        kfsd_finish_kernel<<<(unsigned)ceil_div(rows, 256), 256, 0, st>>>(pa, pb, pq, rows, ntile, d_r + r0);
        ctx->last.launches += 3;
        SD_CUDA(cudaGetLastError());
    }
    return SD_OK;
}

}  // namespace sd
