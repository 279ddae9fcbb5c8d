// outliers.cu -- the per-curve quantities of functional outlier detection (K8).
//
// Rank sums (outliergram, boxplot ordering).  With b_t / a_t the other curves strictly below / above curve c at
// row t (the integers K1 ranks with), per curve in int64:
//     Q_c = sum_t [C(n-1,2) - C(b_t,2) - C(a_t,2)]   (the relaxed J = 2 numerator: MBD = Q / T / C(n,2))
//     B_c = sum_t b_t,   A_c = sum_t a_t              (the modified epigraph index is 1 - B / (n T))
// Rank-only passes of the rank pipeline (mbd.cu) fill int32 rank rows in row blocks; rank_sums_kernel then reads
// them coalesced along c, one thread per (curve, RS_ROWS rows), and adds its three partial sums with one int64
// atomic each.  A rank outside 0 <= b, a, b + a <= n - 1 sets ST_INTERNAL (never a trap).
//
// Envelope (functional boxplot).  Per row t, over the curves with member[c] != 0: lo_t = min, hi_t = max (returned),
// and the fences  w = hi - lo,  f = factor * w,  lower_t = lo - f,  upper_t = hi + f,  each one correctly rounded
// double operation (no FMA: the file is built with -fmad=false and the ops are spelled __d*_rn), so the host
// rebuilds the very fences the counts were taken against; outside[c] counts the rows with x < lower or x > upper.
//   envelope_minmax_kernel  grid (T, chunks): masked min / max of one row chunk, folded into the row's two slots
//                           as order-preserving u64 keys with one atomicMin / atomicMax per CTA.  Also the
//                           finite check of every value.
//   envelope_fences_kernel  grid (T, chunks) when counting, (T, 1) otherwise: block (t, 0) stores lo / hi; with
//                           counts, every block forms the fences, re-reads its chunk and bumps a curve's counter
//                           only on a hit (outside values are rare).
// Shape: T >= 4 * #SMs rows (T = 1024 at 148 SMs is 1024 CTAs of 800 KB rows at n = 100 000) leaves one CTA per
// row.  Small T with huge n splits every row into chunks of at least ENV_MIN_CHUNK curves so that T * chunks
// reaches 4 * #SMs CTAs (T = 1, n = 10^7: 592 CTAs of 16 900 curves); the key atomics make the split free of a
// second reduction launch.  Counting re-reads X (from L2 only when X fits there): the floor is two reads of X.
#include "common.cuh"

namespace sd {

constexpr int RS_THREADS = 256;
constexpr int RS_ROWS = 32;        // rank rows summed per thread before its atomics
constexpr i64 RS_MAX_ROW_TILES = 65535;  // gridDim.y

__global__ void __launch_bounds__(RS_THREADS) rank_sums_kernel(const int *__restrict__ rb, const int *__restrict__ ra,
                                                               const i64 n, const i64 rows, i64 *__restrict__ q,
                                                               i64 *__restrict__ bsum, i64 *__restrict__ asum,
                                                               int *__restrict__ status) {
    const i64 c = (i64)blockIdx.x * RS_THREADS + threadIdx.x;
    if (c >= n) return;
    const i64 r0 = (i64)blockIdx.y * RS_ROWS;
    const i64 r1 = r0 + RS_ROWS < rows ? r0 + RS_ROWS : rows;
    const i64 full = (n - 1) * (n - 2) / 2;
    i64 sq = 0, sb = 0, sa = 0;
    bool bad = false;
    for (i64 r = r0; r < r1; ++r) {
        const i64 b = rb[r * n + c], a = ra[r * n + c];
        if (b < 0 || a < 0 || b + a > n - 1) {
            bad = true;
            continue;
        }
        sq += full - b * (b - 1) / 2 - a * (a - 1) / 2;
        sb += b;
        sa += a;
    }
    if (bad) atomicOr(status, ST_INTERNAL);
    if (sq) atomicAdd((u64 *)&q[c], (u64)sq);
    if (sb) atomicAdd((u64 *)&bsum[c], (u64)sb);
    if (asum && sa) atomicAdd((u64 *)&asum[c], (u64)sa);
}

int rank_sums_device(sd_ctx *ctx, const double *dX, i64 T, i64 n, i64 ld, i64 *d_q, i64 *d_b, i64 *d_a) {
    if (T < 1 || n < 1 || ld < n) {
        set_error("rank sums: bad shape T=%lld n=%lld ld=%lld", (long long)T, (long long)n, (long long)ld);
        return SD_ERR_INVALID;
    }
    SD_TRY(relaxed_overflow_check(T, n - 1, 2, "rank sums"));  // the J = 2 numerator; B and A are smaller
    cudaStream_t st = ctx->stream;
    SD_CUDA(cudaMemsetAsync(d_q, 0, (size_t)n * sizeof(i64), st));
    SD_CUDA(cudaMemsetAsync(d_b, 0, (size_t)n * sizeof(i64), st));
    if (d_a) SD_CUDA(cudaMemsetAsync(d_a, 0, (size_t)n * sizeof(i64), st));
    return for_each_rank_block(ctx, dX, T, n, ld, true, RS_MAX_ROW_TILES * RS_ROWS,
                               [&](i64, i64 rows, const int *rb, const int *ra) {
        const dim3 grid((unsigned)ceil_div(n, RS_THREADS), (unsigned)ceil_div(rows, RS_ROWS));
        rank_sums_kernel<<<grid, RS_THREADS, 0, st>>>(rb, ra, n, rows, d_q, d_b, d_a, ctx->d_status);
        ctx->last.launches++;
    });
}

constexpr int ENV_THREADS = 256;
constexpr int ENV_UNROLL = 4;        // independent loads in flight per thread
constexpr i64 ENV_MIN_CHUNK = 4096;  // curves per CTA at least, when rows are split
constexpr i64 ENV_MAX_CHUNKS = 65535;  // gridDim.y

__device__ __forceinline__ double key_to_double(const u64 k) {
    return __longlong_as_double((long long)((k >> 63) ? (k ^ 0x8000000000000000ull) : ~k));
}

// keys[t] = min key, keys[T + t] = max key of row t (initialised to ~0 / 0: min > max means no member seen)
__global__ void __launch_bounds__(ENV_THREADS) envelope_minmax_kernel(const double *__restrict__ X, const i64 T,
                                                                      const i64 n, const i64 ld, const i64 chunk,
                                                                      const uint8_t *__restrict__ member,
                                                                      u64 *__restrict__ keys,
                                                                      int *__restrict__ status) {
    const i64 t = blockIdx.x;
    const i64 c0 = (i64)blockIdx.y * chunk;
    const i64 c1 = c0 + chunk < n ? c0 + chunk : n;
    const double *row = X + t * ld;
    u64 kmin = ~0ull, kmax = 0;
    bool bad = false;
    for (i64 c = c0 + threadIdx.x; c < c1; c += ENV_THREADS * ENV_UNROLL) {
        double v[ENV_UNROLL];
        uint8_t m[ENV_UNROLL];
#pragma unroll
        for (int u = 0; u < ENV_UNROLL; ++u) {
            const i64 cc = c + u * ENV_THREADS;
            v[u] = cc < c1 ? row[cc] : 0.0;
            m[u] = cc < c1 ? member[cc] : 0;
        }
#pragma unroll
        for (int u = 0; u < ENV_UNROLL; ++u) {
            bad |= !isfinite(v[u]);
            if (m[u]) {
                const u64 k = sortable_key(v[u]);
                kmin = k < kmin ? k : kmin;
                kmax = k > kmax ? k : kmax;
            }
        }
    }
    if (bad) atomicOr(status, ST_NONFINITE);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const u64 omin = __shfl_xor_sync(0xffffffffu, kmin, o), omax = __shfl_xor_sync(0xffffffffu, kmax, o);
        kmin = omin < kmin ? omin : kmin;
        kmax = omax > kmax ? omax : kmax;
    }
    __shared__ u64 smin[ENV_THREADS / 32], smax[ENV_THREADS / 32];
    const int w = threadIdx.x >> 5;
    if ((threadIdx.x & 31) == 0) {
        smin[w] = kmin;
        smax[w] = kmax;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int k = 1; k < ENV_THREADS / 32; ++k) {
            kmin = smin[k] < kmin ? smin[k] : kmin;
            kmax = smax[k] > kmax ? smax[k] : kmax;
        }
        if (kmin <= kmax) {  // this chunk holds a member
            atomicMin(&keys[t], kmin);
            atomicMax(&keys[T + t], kmax);
        }
    }
}

template <bool COUNT>
__global__ void __launch_bounds__(ENV_THREADS) envelope_fences_kernel(const double *__restrict__ X, const i64 T,
                                                                      const i64 n, const i64 ld, const i64 chunk,
                                                                      const u64 *__restrict__ keys, const double factor,
                                                                      double *__restrict__ lower,
                                                                      double *__restrict__ upper,
                                                                      i64 *__restrict__ outside,
                                                                      int *__restrict__ status) {
    const i64 t = blockIdx.x;
    const u64 kmin = keys[t], kmax = keys[T + t];
    const bool lead = blockIdx.y == 0 && threadIdx.x == 0;
    if (kmin > kmax) {
        if (lead) atomicOr(status, ST_NO_MEMBER);
        return;
    }
    const double lo = key_to_double(kmin), hi = key_to_double(kmax);
    if (lead) {
        lower[t] = lo;
        upper[t] = hi;
    }
    if (!COUNT) return;
    const double f = __dmul_rn(factor, __dsub_rn(hi, lo));
    const double lf = __dsub_rn(lo, f), uf = __dadd_rn(hi, f);
    const i64 c0 = (i64)blockIdx.y * chunk;
    const i64 c1 = c0 + chunk < n ? c0 + chunk : n;
    const double *row = X + t * ld;
    for (i64 c = c0 + threadIdx.x; c < c1; c += ENV_THREADS * ENV_UNROLL) {
        double v[ENV_UNROLL];
#pragma unroll
        for (int u = 0; u < ENV_UNROLL; ++u) {
            const i64 cc = c + u * ENV_THREADS;
            v[u] = cc < c1 ? row[cc] : lf;
        }
#pragma unroll
        for (int u = 0; u < ENV_UNROLL; ++u)
            if (v[u] < lf || v[u] > uf) atomicAdd((u64 *)&outside[c + u * ENV_THREADS], 1ull);
    }
}

int envelope_device(sd_ctx *ctx, const double *dX, i64 T, i64 n, i64 ld, const uint8_t *d_member, double factor,
                    double *d_lower, double *d_upper, i64 *d_outside) {
    if (T < 1 || n < 1 || ld < n) {
        set_error("envelope: bad shape T=%lld n=%lld ld=%lld", (long long)T, (long long)n, (long long)ld);
        return SD_ERR_INVALID;
    }
    if (!(factor >= 0.0 && factor <= 1.7976931348623157e308)) {
        set_error("envelope: factor must be finite and >= 0");
        return SD_ERR_INVALID;
    }
    cudaStream_t st = ctx->stream;
    i64 chunks = ceil_div(4 * (i64)ctx->sm_count, T);
    const i64 most = ceil_div(n, ENV_MIN_CHUNK);
    if (chunks > most) chunks = most;
    if (chunks > ENV_MAX_CHUNKS) chunks = ENV_MAX_CHUNKS;
    const i64 chunk = ceil_div(n, chunks);
    SD_TRY(ctx->buf[BUF_AUX].reserve((size_t)2 * T * sizeof(u64)));
    u64 *keys = ctx->buf[BUF_AUX].as<u64>();
    SD_CUDA(cudaMemsetAsync(keys, 0xff, (size_t)T * sizeof(u64), st));
    SD_CUDA(cudaMemsetAsync(keys + T, 0, (size_t)T * sizeof(u64), st));
    if (d_outside) SD_CUDA(cudaMemsetAsync(d_outside, 0, (size_t)n * sizeof(i64), st));
    envelope_minmax_kernel<<<dim3((unsigned)T, (unsigned)chunks), ENV_THREADS, 0, st>>>(dX, T, n, ld, chunk, d_member,
                                                                                      keys, ctx->d_status);
    ctx->last.launches++;
    SD_CUDA(cudaGetLastError());
    if (d_outside)
        envelope_fences_kernel<true><<<dim3((unsigned)T, (unsigned)chunks), ENV_THREADS, 0, st>>>(
            dX, T, n, ld, chunk, keys, factor, d_lower, d_upper, d_outside, ctx->d_status);
    else
        envelope_fences_kernel<false><<<dim3((unsigned)T, 1), 32, 0, st>>>(dX, T, n, ld, chunk, keys, factor, d_lower,
                                                                          d_upper, nullptr, ctx->d_status);
    ctx->last.launches++;
    SD_CUDA(cudaGetLastError());
    return SD_OK;
}

}  // namespace sd
