// spatial.cu -- functional spatial depth (K14): a curve is the vector of its F = T d values and
//   r_q = || sum_{j : x_j != x_q} (x_j - x_q) / ||x_j - x_q|| ||,   depth = 1 - r_q / n_pop (formed by the host).
//
// Two GEMM-shaped passes over (query tile x sample tile) blocks on the FP64 pipe (tcgen05.mma has no f64 kind), both
// streaming their reduction dimension through shared memory in double-buffered cp.async chunks:
//   distance pass  W[q][s] = 1 / sqrt(sum_f (x_q,f - x_s,f)^2), 0 for a zero distance (the query itself, duplicates,
//                  differences that underflow); a squared distance that overflows sets ST_OVERFLOW;
//   sum pass       S_q,f = sum_s W[q][s] (x_s,f - x_q,f) in this direct-difference form (W X - (sum_s W) x_q would
//                  cancel catastrophically far from the origin), then ||S_q||^2 per block of features, then r_q.
// Every query's sums run in an order fixed by the indices and the tile sizes alone (each thread walks f, resp. s, in
// order; the feature blocks are added in order): no float atomics, and a query's r does not depend on the other
// queries, the row block or the number of queries.  Zero weights add exact zeros, so the sample with the query
// appended (in-sample) and the sample alone (out of sample) give the same bits.
#include <float.h>

#include "common.cuh"

namespace sd {

constexpr int SP_THREADS = 256;      // 16 x 16 threads
constexpr int SP_TQ = 4;             // register micro-tile: queries ...
constexpr int SP_TS = 8;             // ... x samples (distance pass) or x features (sum pass), strided by 16
constexpr int SP_BQ = 16 * SP_TQ;    // 64 queries per block
constexpr int SP_BS = 16 * SP_TS;    // 128 samples / features per block
constexpr int SP_BK = 16;            // reduction chunk staged in shared memory
constexpr size_t SP_W_BUDGET = 1ull << 30;  // bytes of one W row block (BUF_SPATIAL)

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

// grid (ceil(nS / SP_BS), ceil(nq / SP_BQ)).  Queries: rows Q[idx(q) * F] (idx = qidx or q); W [nq][nS].
__global__ void __launch_bounds__(SP_THREADS) spatial_dist_kernel(const double *__restrict__ Q,
                                                                  const i64 *__restrict__ qidx, const i64 nq,
                                                                  const double *__restrict__ S, const i64 nS,
                                                                  const i64 F, double *__restrict__ W,
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
    bool overflow = false;
#pragma unroll
    for (int i = 0; i < SP_TQ; ++i) {
        const i64 q = q0 + ty + 16 * i;
        if (q >= nq) continue;
#pragma unroll
        for (int j = 0; j < SP_TS; ++j) {
            const i64 s = s0 + tx + 16 * j;
            if (s >= nS) continue;
            const double d2 = acc[i][j];
            double w = 0.0;
            if (!(d2 <= DBL_MAX)) overflow = true;  // +inf (or NaN from non-finite input, reported as such)
            else if (d2 > 0.0) w = __drcp_rn(__dsqrt_rn(d2));
            W[q * nS + s] = w;
        }
    }
    if (overflow) atomicOr(status, ST_OVERFLOW);
}

// grid (ceil(F / SP_BS), ceil(nq / SP_BQ)).  part[q * gridDim.x + blockIdx.x] = sum over this block's features f of
// S_q,f^2, S_q,f = sum_s W[q][s] (S[s][f] - Q[idx(q)][f]) accumulated in s order.
__global__ void __launch_bounds__(SP_THREADS, 1) spatial_sum_kernel(const double *__restrict__ Q,
                                                                    const i64 *__restrict__ qidx, const i64 nq,
                                                                    const double *__restrict__ S, const i64 nS,
                                                                    const i64 F, const double *__restrict__ W,
                                                                    double *__restrict__ part) {
    __shared__ __align__(16) double Ws[2][SP_BK][SP_BQ];
    __shared__ __align__(16) double Xs[2][SP_BK][SP_BS];
    const int tx = threadIdx.x % 16, ty = threadIdx.x / 16;
    const i64 q0 = (i64)blockIdx.y * SP_BQ, f0 = (i64)blockIdx.x * SP_BS;
    double xq[SP_TQ][SP_TS], acc[SP_TQ][SP_TS];
#pragma unroll
    for (int i = 0; i < SP_TQ; ++i) {
        const i64 q = q0 + ty + 16 * i;
        const double *row = q < nq ? Q + (qidx ? qidx[q] : q) * F : Q;
#pragma unroll
        for (int j = 0; j < SP_TS; ++j) {
            const i64 f = f0 + tx + 16 * j;
            xq[i][j] = (q < nq && f < F) ? row[f] : 0.0;
            acc[i][j] = 0.0;
        }
    }
    const i64 nk = ceil_div(nS, SP_BK);
    stage_t<SP_BQ>(Ws[0], W, nullptr, q0, nq, nS, 0, nS);
    stage_n<SP_BS>(Xs[0], S, 0, nS, F, f0, F);
    cp_async_commit();
    for (i64 kc = 0; kc < nk; ++kc) {
        const int b = (int)(kc & 1);
        if (kc + 1 < nk) {
            stage_t<SP_BQ>(Ws[b ^ 1], W, nullptr, q0, nq, nS, (kc + 1) * SP_BK, nS);
            stage_n<SP_BS>(Xs[b ^ 1], S, (kc + 1) * SP_BK, nS, F, f0, F);
        }
        cp_async_commit();
        cp_async_wait1();
        __syncthreads();
#pragma unroll
        for (int k = 0; k < SP_BK; ++k) {
            double w[SP_TQ], x[SP_TS];
#pragma unroll
            for (int i = 0; i < SP_TQ; ++i) w[i] = Ws[b][k][(ty + 16 * i) ^ k];
#pragma unroll
            for (int j = 0; j < SP_TS; ++j) x[j] = Xs[b][k][tx + 16 * j];
#pragma unroll
            for (int i = 0; i < SP_TQ; ++i)
#pragma unroll
                for (int j = 0; j < SP_TS; ++j) acc[i][j] = __fma_rn(w[i], __dsub_rn(x[j], xq[i][j]), acc[i][j]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < SP_TQ; ++i) {
        double v = 0.0;
#pragma unroll
        for (int j = 0; j < SP_TS; ++j) v = __fma_rn(acc[i][j], acc[i][j], v);
        // the 16 lanes of one ty: a fixed butterfly, every lane ends with the same bits
#pragma unroll
        for (int m = 1; m < 16; m <<= 1) v = __dadd_rn(v, __shfl_xor_sync(0xffffffffu, v, m));
        const i64 q = q0 + ty + 16 * i;
        if (tx == 0 && q < nq) part[q * gridDim.x + blockIdx.x] = v;
    }
}

__global__ void spatial_norm_kernel(const double *__restrict__ part, const i64 nq, const i64 nfb,
                                    double *__restrict__ r) {
    const i64 q = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= nq) return;
    double v = 0.0;
    for (i64 b = 0; b < nfb; ++b) v = __dadd_rn(v, part[q * nfb + b]);
    r[q] = __dsqrt_rn(v);
}

// r of the nq queries (rows dQ[idx(q) * F], idx = d_qidx or q) against the nS sample rows dS [nS, F]; a query that is
// itself a sample row has distance 0 to it and weight 0.  Row blocks of queries keep W within SP_W_BUDGET.
int spatial_device(sd_ctx *ctx, const double *dQ, const i64 *d_qidx, i64 nq, const double *dS, i64 nS, i64 F,
                   double *d_r) {
    if (nq == 0) return SD_OK;
    const i64 nfb = ceil_div(F, SP_BS);
    i64 RB = (i64)(SP_W_BUDGET / ((size_t)nS * sizeof(double))) / SP_BQ * SP_BQ;
    if (RB < SP_BQ) RB = SP_BQ;
    if (RB > 65535ll * SP_BQ) RB = 65535ll * SP_BQ;  // grid.y
    if (RB > ceil_div(nq, SP_BQ) * SP_BQ) RB = ceil_div(nq, SP_BQ) * SP_BQ;
    SD_TRY(ctx->buf[BUF_SPATIAL].reserve((size_t)RB * (nS + nfb) * sizeof(double)));
    double *dW = ctx->buf[BUF_SPATIAL].as<double>();
    double *dPart = dW + (size_t)RB * nS;
    cudaStream_t st = ctx->stream;
    for (i64 r0 = 0; r0 < nq; r0 += RB) {
        const i64 rows = nq - r0 < RB ? nq - r0 : RB;
        const double *Q = d_qidx ? dQ : dQ + r0 * F;
        const i64 *qi = d_qidx ? d_qidx + r0 : nullptr;
        const unsigned gy = (unsigned)ceil_div(rows, SP_BQ);
        spatial_dist_kernel<<<dim3((unsigned)ceil_div(nS, SP_BS), gy), SP_THREADS, 0, st>>>(Q, qi, rows, dS, nS, F,
                                                                                             dW, ctx->d_status);
        spatial_sum_kernel<<<dim3((unsigned)nfb, gy), SP_THREADS, 0, st>>>(Q, qi, rows, dS, nS, F, dW, dPart);
        spatial_norm_kernel<<<(unsigned)ceil_div(rows, 256), 256, 0, st>>>(dPart, rows, nfb, d_r + r0);
        ctx->last.launches += 3;
        SD_CUDA(cudaGetLastError());
    }
    return SD_OK;
}

}  // namespace sd
