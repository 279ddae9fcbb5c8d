// oos.cu -- out-of-sample band depth: the depth of new curves Y against a reference sample S, every new curve
// counted as if it alone were appended to S (what the reference returns for g after pd.concat([S, g])).
//
// Inputs are one pooled matrix X[t*ld + c]: columns [0, nS) the sample, [nS, nS + nY) the new curves.
//
// Relaxed (MBD).  The numerator of new curve g is  sum_t [C(nS,j) - C(b_t,j) - C(a_t,j)],  b_t / a_t the sample
// curves strictly below / above g(t).  Two rank-only passes of the rank pipeline (mbd.cu) give them exactly:
//     pooled pass (n = nS + nY):  bP = #S below + #Y below,     Y pass (n = nY):  bY = #Y below
// so b = bP - bY (and a likewise).  Ties among new curves fall out of both counts; a tie with g is in neither.
// oos_terms_kernel forms the differences, checks 0 <= b, a and b + a <= nS (a failure sets ST_INTERNAL, it never
// traps), and sums the j-term per curve in int64.  Cost: two rank passes over T (nS + 2 nY) values instead of nY
// rank passes over T (nS + 1).
//
// Strict.  The unchanged bit-mask kernels of bd_bits.cu already take "the m = n - 1 others, skipping the query":
// called with n = nS + 1 on the pooled matrix and query ids nS + g >= nS, no other is ever skipped, so the others
// are exactly the sample columns and the query values are read from Y.
#include "common.cuh"

namespace sd {

__global__ void iota_from_kernel(i64 *__restrict__ p, const i64 count, const i64 base) {
    const i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < count) p[i] = base + i;
}

// ST_NONFINITE if any of rows x cols values (leading dimension ld) is NaN or +-inf
__global__ void finite_check_kernel(const double *__restrict__ X, const i64 rows, const i64 cols, const i64 ld,
                                    int *__restrict__ status) {
    bool bad = false;
    const i64 total = rows * cols;
    for (i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (i64)gridDim.x * blockDim.x)
        bad |= !isfinite(X[(i / cols) * ld + i % cols]);
    if (bad) atomicOr(status, ST_NONFINITE);
}

int iota_from_device(sd_ctx *ctx, i64 *d_p, i64 count, i64 base) {
    if (count == 0) return SD_OK;
    iota_from_kernel<<<(unsigned)ceil_div(count, 256), 256, 0, ctx->stream>>>(d_p, count, base);
    ctx->last.launches++;
    SD_CUDA(cudaGetLastError());
    return SD_OK;
}

int finite_check_device(sd_ctx *ctx, const double *dX, i64 rows, i64 cols, i64 ld) {
    if (rows == 0 || cols == 0) return SD_OK;
    i64 grid = ceil_div(rows * cols, 256);
    if (grid > 4 * (i64)ctx->sm_count) grid = 4 * (i64)ctx->sm_count;
    finite_check_kernel<<<(unsigned)grid, 256, 0, ctx->stream>>>(dX, rows, cols, ld, ctx->d_status);
    ctx->last.launches++;
    SD_CUDA(cudaGetLastError());
    return SD_OK;
}

constexpr int OOS_THREADS = 256;
constexpr int OOS_ROWS = 32;  // time rows summed per thread before its one atomic

// grid (new-curve tiles, row tiles).  One thread per (new curve g, OOS_ROWS rows): the rank rows are read
// coalesced along g.  bY / aY == nullptr: a single new curve (no other new curve to subtract).
template <int J>
__global__ void __launch_bounds__(OOS_THREADS) oos_terms_kernel(const int *__restrict__ bP, const int *__restrict__ aP,
                                                                const int *__restrict__ bY, const int *__restrict__ aY,
                                                                const i64 nS, const i64 nY, const i64 rows,
                                                                i64 *__restrict__ acc, int *__restrict__ status) {
    const i64 g = (i64)blockIdx.x * OOS_THREADS + threadIdx.x;
    if (g >= nY) return;
    const i64 n = nS + nY;
    const i64 r0 = (i64)blockIdx.y * OOS_ROWS;
    const i64 r1 = r0 + OOS_ROWS < rows ? r0 + OOS_ROWS : rows;
    const i64 full = oos_comb(nS, J);
    i64 sum = 0;
    bool bad = false;
    for (i64 r = r0; r < r1; ++r) {
        i64 b = bP[r * n + nS + g], a = aP[r * n + nS + g];
        if (bY) {
            b -= bY[r * nY + g];
            a -= aY[r * nY + g];
        }
        if (b < 0 || a < 0 || b + a > nS) {
            bad = true;
            continue;
        }
        sum += full - oos_comb(b, J) - oos_comb(a, J);
    }
    if (bad) atomicOr(status, ST_INTERNAL);
    if (sum) atomicAdd((u64 *)&acc[g], (u64)sum);
}

int band_depth_oos_device(sd_ctx *ctx, const double *dX, i64 T, i64 nS, i64 nY, i64 ld, int j, int relax,
                          i64 *d_out) {
    if (j != 2 && j != 3) {
        set_error("out-of-sample band depth: subset size j=%d not supported on the device (2 or 3)", j);
        return SD_ERR_UNSUPPORTED;
    }
    if (T < 1 || nS < 1 || nY < 0 || ld < nS + nY) {
        set_error("out-of-sample band depth: bad shape T=%lld nS=%lld nY=%lld ld=%lld", (long long)T, (long long)nS,
                  (long long)nY, (long long)ld);
        return SD_ERR_INVALID;
    }
    cudaStream_t st = ctx->stream;
    SD_CUDA(cudaMemsetAsync(d_out, 0, (size_t)(nY > 0 ? nY : 1) * sizeof(i64), st));
    if (nY == 0) return SD_OK;
    if (!relax) {
        // the mask kernel checks the others (and the first new curve); the remaining query values here
        SD_TRY(finite_check_device(ctx, dX + nS, T, nY, ld));
        SD_TRY(ctx->buf[BUF_QIDX].reserve((size_t)nY * sizeof(i64)));
        i64 *d_q = ctx->buf[BUF_QIDX].as<i64>();
        SD_TRY(iota_from_device(ctx, d_q, nY, nS));
        ctx->last.bd_impl_used = SD_BD_BITS;
        return bd_strict_device(ctx, dX, T, nS + 1, ld, d_q, nY, j, d_out);
    }
    SD_TRY(relaxed_overflow_check(T, nS, j, "out-of-sample band depth"));
    const i64 n = nS + nY;
    const i64 ny_ranks = nY > 1 ? nY : 0;  // one new curve: nothing to subtract, no second pass
    i64 RB = 0;
    int *bP = nullptr;
    SD_TRY(rank_block_workspace(ctx, T, (n + ny_ranks) * 2, &RB, &bP));
    int *aP = bP + (size_t)RB * n;
    int *bY = ny_ranks ? aP + (size_t)RB * n : nullptr;
    int *aY = ny_ranks ? bY + (size_t)RB * nY : nullptr;
    for (i64 r0 = 0; r0 < T; r0 += RB) {
        const i64 rows = T - r0 < RB ? T - r0 : RB;
        const double *Xb = dX + r0 * ld;
        SD_TRY(rank_rows_device(ctx, Xb, rows, n, ld, bP, aP));
        if (ny_ranks) SD_TRY(rank_rows_device(ctx, Xb + nS, rows, nY, ld, bY, aY));
        const dim3 grid((unsigned)ceil_div(nY, OOS_THREADS), (unsigned)ceil_div(rows, OOS_ROWS));
        if (j == 2) oos_terms_kernel<2><<<grid, OOS_THREADS, 0, st>>>(bP, aP, bY, aY, nS, nY, rows, d_out, ctx->d_status);
        else oos_terms_kernel<3><<<grid, OOS_THREADS, 0, st>>>(bP, aP, bY, aY, nS, nY, rows, d_out, ctx->d_status);
        ctx->last.launches++;
        SD_CUDA(cudaGetLastError());
    }
    return SD_OK;
}

}  // namespace sd
