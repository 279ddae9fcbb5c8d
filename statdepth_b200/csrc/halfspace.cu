// halfspace.cu -- halfspace (Tukey) depth numerators of univariate values (K11, d = 1).
//
// With b_t / a_t the other curves strictly below / above curve c at row t (the integers K1 ranks with), the closed
// half-lines through c(t) hold #{x <= c(t)} = n - a_t and #{x >= c(t)} = n - b_t values, c itself included, so
//     H_c = sum_t h_t(c),   h_t(c) = min(n - a_t, n - b_t) = n - max(b_t, a_t)   in [1, n]
// (a point cloud of dimension 1 is one row, T = 1).  As rank_sums_kernel (outliers.cu): rank-only passes of the rank
// pipeline fill int32 rank rows in row blocks, one thread per (curve, HS_ROWS rows) adds its partial sum with one
// int64 atomic.  A rank outside 0 <= b, a, b + a <= n - 1 sets ST_INTERNAL (never a trap).  The 2-D form is
// hs_reduce_kernel (simplicial_count.cu).
#include "common.cuh"

namespace sd {

constexpr int HS_THREADS = 256;
constexpr int HS_ROWS = 32;               // rank rows summed per thread before its atomic
constexpr i64 HS_MAX_ROW_TILES = 65535;   // gridDim.y

__global__ void __launch_bounds__(HS_THREADS) halfspace_terms_kernel(const int *__restrict__ rb,
                                                                     const int *__restrict__ ra, const i64 n,
                                                                     const i64 rows, i64 *__restrict__ out,
                                                                     int *__restrict__ status) {
    const i64 c = (i64)blockIdx.x * HS_THREADS + threadIdx.x;
    if (c >= n) return;
    const i64 r0 = (i64)blockIdx.y * HS_ROWS;
    const i64 r1 = r0 + HS_ROWS < rows ? r0 + HS_ROWS : rows;
    i64 s = 0;
    bool bad = false;
    for (i64 r = r0; r < r1; ++r) {
        const i64 b = rb[r * n + c], a = ra[r * n + c];
        if (b < 0 || a < 0 || b + a > n - 1) {
            bad = true;
            continue;
        }
        s += n - (b > a ? b : a);
    }
    if (bad) atomicOr(status, ST_INTERNAL);
    if (s) atomicAdd((u64 *)&out[c], (u64)s);
}

int halfspace1_device(sd_ctx *ctx, const double *dX, i64 T, i64 n, i64 ld, i64 *d_out) {
    if (T < 1 || n < 1 || ld < n) {
        set_error("halfspace depth: bad shape T=%lld n=%lld ld=%lld", (long long)T, (long long)n, (long long)ld);
        return SD_ERR_INVALID;
    }
    cudaStream_t st = ctx->stream;
    SD_CUDA(cudaMemsetAsync(d_out, 0, (size_t)n * sizeof(i64), st));
    return for_each_rank_block(ctx, dX, T, n, ld, true, HS_MAX_ROW_TILES * HS_ROWS,
                               [&](i64, i64 rows, const int *rb, const int *ra) {
        const dim3 grid((unsigned)ceil_div(n, HS_THREADS), (unsigned)ceil_div(rows, HS_ROWS));
        halfspace_terms_kernel<<<grid, HS_THREADS, 0, st>>>(rb, ra, n, rows, d_out, ctx->d_status);
        ctx->last.launches++;
    });
}

}  // namespace sd
