// reference.cu -- a reference sample indexed once on the device, new curves scored against it by binary search (K9).
//
// Relaxed out-of-sample band depth (oos.cu) needs, per new curve g and row t, only b_t / a_t: the sample values
// strictly below / above g(t).  Both are binary searches in the sorted row t of the sample, so a reference that is
// scored against again and again is sorted once and kept on the device; each later call reads only the new curves.
//
// Build (sort_rows_device): sorted[t*nS + k] = the k-th smallest of row t, ties repeated.
//   1. K1 rank-only passes in row blocks (for_each_rank_block, mbd.cu) give every value its below-rank b (exact,
//      finite check included).
//   2. sort_scatter_kernel  sorted[t][b] = X[t, c].  All curves of a tie run share b and write equal values to the
//                           run's first slot (benign race; -0.0 and +0.0 compare equal, either may land).  The other
//                           slots of the run keep the gap sentinel the rows were filled with before: an all-ones NaN
//                           (cudaMemsetAsync writes it at copy rate; the input is finite, so a NaN is never a value).
//   3. sort_fill_kernel     grid (T, chunks): one CTA per row chunk carries the last value over the gaps with a
//                           block-wide scan and writes only the gaps, so tie-free rows are read once and not written.
//                           A chunk finds its carry-in by searching backwards from its first slot (slot 0 of a row
//                           always holds a value: the row minimum has b = 0).
//
// Query (depth_sorted_device): count[(j-2)*nY + g] = sum_t [C(nS,j) - C(b_t,j) - C(a_t,j)], j = 2..J, equal to
// band_depth_oos_device(relax = 1, j).  sorted_terms_kernel: one thread per (new curve g, block of R rows), Y read
// coalesced along g; per row sorted_bounds (sorted_row.cuh): a lower and an upper bound search of y in the same loop
// (their step sizes depend on nS only, so the two chains of dependent loads interleave and no warp diverges).  Every
// index read stays in [0, nS)
// and every result in [0, nS] whatever the buffer holds; 0 <= b, a and b + a <= nS is checked all the same (a
// failure sets ST_INTERNAL, the kernel never traps).  One int64 atomic per (g, row block, j).
// R is 32 rows when there are enough new curves to fill the GPU; fewer new curves get fewer rows per thread, down to
// one, so that n_Y * T / R threads still reach ~ 2 full occupancies (each row costs ~2 log2(nS) dependent loads).
#include "sorted_row.cuh"

namespace sd {

constexpr int SORT_THREADS = 256;
constexpr i64 SORT_MAX_ROWS = 65535;  // gridDim.y of the scatter
constexpr int FILL_THREADS = 256;
constexpr int FILL_VALS = 4;                           // contiguous slots per thread per tile
constexpr i64 FILL_TILE = FILL_THREADS * FILL_VALS;
constexpr i64 FILL_MIN_CHUNK = 4096;                    // slots per CTA at least, when rows are split
constexpr i64 FILL_MAX_CHUNKS = 65535;                  // gridDim.y
constexpr int Q_THREADS = 256;
constexpr i64 Q_MAX_ROWS = 32;      // rows per thread when n_Y is large
constexpr i64 Q_MAX_ROW_TILES = 65535;  // gridDim.y

__device__ __forceinline__ bool is_gap(const double v) { return v != v; }

__global__ void __launch_bounds__(SORT_THREADS) sort_scatter_kernel(const double *__restrict__ X, const i64 ld,
                                                                    const int *__restrict__ below, const i64 nS,
                                                                    double *__restrict__ sorted,
                                                                    int *__restrict__ status) {
    const i64 c = (i64)blockIdx.x * SORT_THREADS + threadIdx.x;
    if (c >= nS) return;
    const i64 r = blockIdx.y;
    const int b = below[r * nS + c];
    if (b < 0 || b >= nS) {
        atomicOr(status, ST_INTERNAL);
        return;
    }
    sorted[r * nS + b] = X[r * ld + c];
}

// the last value (not a gap) of v, gap if none: x = last(v[0..k]) combined left to right keeps the right operand
// unless it is a gap
__device__ __forceinline__ double keep_last(const double left, const double right) {
    return is_gap(right) ? left : right;
}

__global__ void __launch_bounds__(FILL_THREADS) sort_fill_kernel(double *__restrict__ sorted, const i64 nS,
                                                                 const i64 chunk, int *__restrict__ status) {
    __shared__ long long found;
    __shared__ double warp_last[FILL_THREADS / 32];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    double *row = sorted + (i64)blockIdx.x * nS;
    const i64 c0 = (i64)blockIdx.y * chunk;
    const i64 c1 = c0 + chunk < nS ? c0 + chunk : nS;
    const double gap = __longlong_as_double(-1ll);
    double carry = gap;
    if (c0 > 0) {  // carry-in: the last value before the chunk
        if (threadIdx.x == 0) found = -1;
        __syncthreads();
        for (i64 e = c0; e > 0; e -= FILL_THREADS) {
            const i64 p = e - 1 - threadIdx.x;
            if (p >= 0 && !is_gap(row[p])) atomicMax(&found, (long long)p);
            __syncthreads();
            const long long f = found;
            __syncthreads();  // every thread has read `found` before the next round may raise it
            if (f >= 0) break;
        }
        if (found >= 0) carry = row[found];
        else if (threadIdx.x == 0) atomicOr(status, ST_INTERNAL);  // slot 0 holds no value
    }
    for (i64 base = c0; base < c1; base += FILL_TILE) {
        const i64 p0 = base + (i64)threadIdx.x * FILL_VALS;
        double v[FILL_VALS];
        double mine = gap;
#pragma unroll
        for (int u = 0; u < FILL_VALS; ++u) {
            v[u] = p0 + u < c1 ? row[p0 + u] : 0.0;  // past the chunk: a value, never written
            if (p0 + u < c1) mine = keep_last(mine, v[u]);
        }
        // inclusive warp scan of the threads' last values, then the warps' last values through shared memory
        double x = mine;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const double y = __shfl_up_sync(0xffffffffu, x, o);
            if (lane >= o) x = keep_last(y, x);
        }
        double before = __shfl_up_sync(0xffffffffu, x, 1);  // exclusive within the warp
        if (lane == 0) before = gap;
        if (lane == 31) warp_last[w] = x;
        __syncthreads();
        double run = carry;
        for (int k = 0; k < w; ++k) run = keep_last(run, warp_last[k]);
        run = keep_last(run, before);
#pragma unroll
        for (int u = 0; u < FILL_VALS; ++u) {
            if (p0 + u >= c1) break;
            if (is_gap(v[u])) {
                if (!is_gap(run)) row[p0 + u] = run;
            } else {
                run = v[u];
            }
        }
        for (int k = 0; k < FILL_THREADS / 32; ++k) carry = keep_last(carry, warp_last[k]);
        __syncthreads();  // warp_last is rewritten by the next tile
    }
}

int sort_rows_device(sd_ctx *ctx, const double *dX, i64 T, i64 nS, i64 ld, double *d_sorted) {
    if (T < 1 || nS < 1 || ld < nS) {
        set_error("sort rows: bad shape T=%lld nS=%lld ld=%lld", (long long)T, (long long)nS, (long long)ld);
        return SD_ERR_INVALID;
    }
    cudaStream_t st = ctx->stream;
    SD_CUDA(cudaMemsetAsync(d_sorted, 0xff, (size_t)T * nS * sizeof(double), st));  // gap sentinel: a NaN
    SD_TRY(for_each_rank_block(ctx, dX, T, nS, ld, false, SORT_MAX_ROWS,
                               [&](i64 r0, i64 rows, const int *below, const int *) {
        sort_scatter_kernel<<<dim3((unsigned)ceil_div(nS, SORT_THREADS), (unsigned)rows), SORT_THREADS, 0, st>>>(
            dX + r0 * ld, ld, below, nS, d_sorted + r0 * nS, ctx->d_status);
        ctx->last.launches++;
    }));
    i64 chunks = ceil_div(4 * (i64)ctx->sm_count, T);
    const i64 most = ceil_div(nS, FILL_MIN_CHUNK);
    if (chunks > most) chunks = most;
    if (chunks > FILL_MAX_CHUNKS) chunks = FILL_MAX_CHUNKS;
    const i64 chunk = ceil_div(nS, chunks);
    sort_fill_kernel<<<dim3((unsigned)T, (unsigned)chunks), FILL_THREADS, 0, st>>>(d_sorted, nS, chunk, ctx->d_status);
    ctx->last.launches++;
    SD_CUDA(cudaGetLastError());
    return SD_OK;
}

// grid (new-curve tiles, row tiles): thread (g, rows [r0, r0 + R)).  acc[(j-2)*nY + g].
template <int J>
__global__ void __launch_bounds__(Q_THREADS) sorted_terms_kernel(const double *__restrict__ sorted, const i64 T,
                                                                 const i64 nS, const double *__restrict__ Y,
                                                                 const i64 nY, const i64 ldY, const i64 R,
                                                                 i64 *__restrict__ acc, int *__restrict__ status) {
    const i64 g = (i64)blockIdx.x * Q_THREADS + threadIdx.x;
    if (g >= nY) return;
    const i64 r0 = (i64)blockIdx.y * R;
    const i64 r1 = r0 + R < T ? r0 + R : T;
    const i64 full2 = oos_comb(nS, 2), full3 = J == 3 ? oos_comb(nS, 3) : 0;
    i64 s2 = 0, s3 = 0;
    bool bad = false;
    for (i64 t = r0; t < r1; ++t) {
        i64 b, a;
        sorted_bounds(sorted + t * nS, nS, Y[t * ldY + g], b, a);
        if (b < 0 || a < 0 || b + a > nS) {
            bad = true;
            continue;
        }
        s2 += full2 - oos_comb(b, 2) - oos_comb(a, 2);
        if (J == 3) s3 += full3 - oos_comb(b, 3) - oos_comb(a, 3);
    }
    if (bad) atomicOr(status, ST_INTERNAL);
    if (s2) atomicAdd((u64 *)&acc[g], (u64)s2);
    if (J == 3 && s3) atomicAdd((u64 *)&acc[nY + g], (u64)s3);
}

int depth_sorted_device(sd_ctx *ctx, const double *d_sorted, i64 T, i64 nS, const double *dY, i64 nY, i64 ldY,
                        int J, i64 *d_out) {
    if (J != 2 && J != 3) {
        set_error("sorted-reference band depth: J=%d not supported on the device (2 or 3)", J);
        return SD_ERR_UNSUPPORTED;
    }
    if (T < 1 || nS < 1 || nY < 0 || ldY < nY) {
        set_error("sorted-reference band depth: bad shape T=%lld nS=%lld nY=%lld ldY=%lld", (long long)T,
                  (long long)nS, (long long)nY, (long long)ldY);
        return SD_ERR_INVALID;
    }
    for (int j = 2; j <= J; ++j) SD_TRY(relaxed_overflow_check(T, nS, j, "sorted-reference band depth"));
    cudaStream_t st = ctx->stream;
    if (nY == 0) return SD_OK;
    SD_CUDA(cudaMemsetAsync(d_out, 0, (size_t)(J - 1) * nY * sizeof(i64), st));
    SD_TRY(finite_check_device(ctx, dY, T, nY, ldY));
    const i64 target = 2 * 2048 * (i64)ctx->sm_count;  // threads for ~2 full occupancies
    i64 R = nY * T / target;
    if (R > Q_MAX_ROWS) R = Q_MAX_ROWS;
    if (R < ceil_div(T, Q_MAX_ROW_TILES)) R = ceil_div(T, Q_MAX_ROW_TILES);
    if (R < 1) R = 1;
    const dim3 grid((unsigned)ceil_div(nY, Q_THREADS), (unsigned)ceil_div(T, R));
    if (J == 2)
        sorted_terms_kernel<2><<<grid, Q_THREADS, 0, st>>>(d_sorted, T, nS, dY, nY, ldY, R, d_out, ctx->d_status);
    else
        sorted_terms_kernel<3><<<grid, Q_THREADS, 0, st>>>(d_sorted, T, nS, dY, nY, ldY, R, d_out, ctx->d_status);
    ctx->last.launches++;
    SD_CUDA(cudaGetLastError());
    return SD_OK;
}

}  // namespace sd
