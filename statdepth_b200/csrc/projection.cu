// projection.cu -- random projection depths (K12): random Tukey depth and projection depth in any dimension.
//
// Data are curves F [N, T, d] (F[(i*T + t)*d + c], a point cloud is T = 1) and directions U [K, d].  Every time
// point t and direction k give one row of N projected values
//     y_k(i, t) = (...((U[k,0] F[i,t,0]) + U[k,1] F[i,t,1]) + ...) + U[k,d-1] F[i,t,d-1]
// summed in this fixed order with correctly rounded products and sums (no FMA; the file is compiled with
// -fmad=false and uses __dmul_rn / __dadd_rn), so that numpy's Y = U0*F0; Y = Y + Uc*Fc gives the same bits.
// Tensor cores are not used: their accumulation order is unspecified, and ties between projections decide ranks.
//
// Random Tukey depth (Cuesta-Albertos & Nieto-Reyes 2008).  With b / a the other values of the row strictly below
// / above y (K1's integers), h_{t,k}(i) = N - max(b, a) in [1, N] (halfspace.cu), and the numerator
//     R(i) = sum_t min_k h_{t,k}(i)   (exact int64, in [T, T*N]);   depth = R / (T N).
// Projection depth (Zuo & Serfling 2000).  Per row, med = np.median and MAD = np.median(|y - med|) (unscaled), and
//     O_t(i) = max_k |y - med| / MAD   (MAD = 0: 0 if y == med, else +inf);   the host forms 1 / (1 + O).
//
// Kernels, per block of rows r = (t, k) (row length N, leading dimension ldY = N rounded up to even so that the
// rank pipeline's slab path can take the rows):
//   projection_kernel   register-tiled like a small GEMM: a CTA computes 128 points x 32 directions, 4 x 4 per
//                       thread, for TT consecutive time points; it stages each point's record of TT * d values
//                       (contiguous in F) through shared memory, or for d > 32 one time point in chunks of 32.
//   RT: rank_rows_device passes (as halfspace1_device), then rt_min_kernel: one thread per (i, up to 32 time
//                       points) reads the block's kb rows of each t coalesced along i and keeps a running int32 min;
//                       after the last direction block it adds sum_t with one int64 atomic.
//   PD: sort_rows_device (K9) into sorted rows, medmad_kernel (one thread per row: row_median / row_mad of
//                       sorted_row.cuh, the median, then the MAD as the k-th smallest of L = |s[m-1..0] - med| and
//                       R = |s[m..] - med|, m = #values < med; both are non-decreasing because rounding is monotone,
//                       so a binary search over how many come from L finds it in O(log N)), then pd_max_kernel: a
//                       running max per (t, i) over the block's rows,
//                       compared as u64 bit patterns (non-negative doubles and +inf order like them).
// Direction blocks continue the running min / max (BUF_PRED), since K N 8 bytes need not fit the workspace (and a
// projection launch takes at most PJ_MAX_KB directions); a time block keeps all K directions whenever K rows fit.
// Y (BUF_PROJ) and the sorted rows (BUF_PSORT) stay within PJ_BUDGET; none of the three slots aliases BUF_RANKS, the
// rank pipeline's buffers or BUF_AUX.
//
// Exactness: F is finite-checked first; a projection that overflows to +-inf (or inf - inf = NaN) is caught by K1's
// finite check in the rank passes (SD_ERR_NONFINITE).  A rank outside 0 <= b, a, b + a <= N - 1 sets ST_INTERNAL
// (never a trap).  Univariate outlyingness (dU == nullptr) skips the projection: the rows of X [T, N] are the
// single direction's rows (u = 1, y = x).
#include "sorted_row.cuh"

namespace sd {

constexpr int PJ_THREADS = 256;
constexpr int PJ_PTS = 128;  // points per CTA, 4 per thread
constexpr int PJ_DIRS = 32;  // directions per CTA, 4 per thread
constexpr int PJ_W = 32;     // record values per point staged per step
constexpr int RD_THREADS = 256;
constexpr i64 RD_MAX_ROWS = 32;  // time points per reduction thread, when there are enough (t, i) pairs
constexpr int MM_THREADS = 128;
constexpr size_t PJ_BUDGET = 1ull << 30;  // bytes of Y (and of the sorted rows) per row block
constexpr i64 PJ_MAX_TB = 65535;          // time points per block (gridDim.z of the projection)
constexpr i64 PJ_MAX_KB = 65535 * PJ_DIRS;  // directions per block (gridDim.y of the projection)

// Y[((tt0 + tt) * kb + kk) * ldY + i] = y_{k0 + kk}(i, t0 + tt0 + tt).  grid (point tiles, direction tiles, time
// tiles of TT); U points at the block's first direction.
__global__ void __launch_bounds__(PJ_THREADS) projection_kernel(const double *__restrict__ F, const i64 N,
                                                                const i64 T, const int d,
                                                                const double *__restrict__ U, const i64 kb,
                                                                const i64 t0, const i64 tb, const int TT,
                                                                double *__restrict__ Y, const i64 ldY) {
    __shared__ double Fs[PJ_PTS][PJ_W + 1];
    __shared__ double Us[PJ_DIRS][PJ_W + 1];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const i64 i0 = (i64)blockIdx.x * PJ_PTS;
    const i64 kk0 = (i64)blockIdx.y * PJ_DIRS;
    const i64 tt0 = (i64)blockIdx.z * TT;
    const int nt = (int)(tb - tt0 < TT ? tb - tt0 : TT);
    for (int tt = 0; tt < nt; ++tt) {
        double acc[4][4];
#pragma unroll
        for (int b = 0; b < 4; ++b)
#pragma unroll
            for (int a = 0; a < 4; ++a) acc[b][a] = -0.0;  // -0 + x == x for every x, -0 included
        for (int c0 = 0; c0 < d; c0 += PJ_W) {
            const int wu = d - c0 < PJ_W ? d - c0 : PJ_W;
            if (tt == 0) {  // d <= PJ_W: the records of all nt time points at once; else this chunk of one
                const int w = d <= PJ_W ? nt * d : wu;
                __syncthreads();
                for (int e = threadIdx.x; e < PJ_PTS * PJ_W; e += PJ_THREADS) {
                    const int p = e / PJ_W, j = e % PJ_W;
                    const i64 i = i0 + p;
                    Fs[p][j] = (i < N && j < w) ? F[(i * T + t0 + tt0) * d + c0 + j] : 0.0;
                }
                for (int e = threadIdx.x; e < PJ_DIRS * PJ_W; e += PJ_THREADS) {
                    const int kk = e / PJ_W, j = e % PJ_W;
                    Us[kk][j] = (kk0 + kk < kb && j < wu) ? U[(kk0 + kk) * d + c0 + j] : 0.0;
                }
                __syncthreads();
            }
            const int fo = d <= PJ_W ? tt * d : 0;
            for (int c = 0; c < wu; ++c) {
                double f[4], u[4];
#pragma unroll
                for (int a = 0; a < 4; ++a) f[a] = Fs[tx + 32 * a][fo + c];
#pragma unroll
                for (int b = 0; b < 4; ++b) u[b] = Us[ty + 8 * b][c];
#pragma unroll
                for (int b = 0; b < 4; ++b)
#pragma unroll
                    for (int a = 0; a < 4; ++a) acc[b][a] = __dadd_rn(acc[b][a], __dmul_rn(u[b], f[a]));
            }
        }
#pragma unroll
        for (int b = 0; b < 4; ++b) {
            const i64 kk = kk0 + ty + 8 * b;
            if (kk >= kb) continue;
            double *row = Y + ((tt0 + tt) * kb + kk) * ldY;
#pragma unroll
            for (int a = 0; a < 4; ++a) {
                const i64 i = i0 + tx + 32 * a;
                if (i < N) row[i] = acc[b][a];
            }
        }
    }
}

// grid (point tiles, time tiles of tpt time points).  Rank rows r = tt * kb + kk, dense with stride N.  run [tb][N].
__global__ void __launch_bounds__(RD_THREADS) rt_min_kernel(const int *__restrict__ rb, const int *__restrict__ ra,
                                                            const i64 N, const i64 kb, const i64 tb, const i64 tpt,
                                                            int *__restrict__ run, const int first, const int last,
                                                            i64 *__restrict__ count, int *__restrict__ status) {
    const i64 i = (i64)blockIdx.x * RD_THREADS + threadIdx.x;
    if (i >= N) return;
    const i64 t0 = (i64)blockIdx.y * tpt;
    const i64 t1 = t0 + tpt < tb ? t0 + tpt : tb;
    i64 s = 0;
    bool bad = false;
    for (i64 t = t0; t < t1; ++t) {
        i64 m = first ? N : run[t * N + i];
        for (i64 kk = 0; kk < kb; ++kk) {
            const i64 r = t * kb + kk;
            const i64 b = rb[r * N + i], a = ra[r * N + i];
            if (b < 0 || a < 0 || b + a > N - 1) {
                bad = true;
                continue;
            }
            const i64 h = N - (b > a ? b : a);
            m = h < m ? h : m;
        }
        if (last) s += m;
        else run[t * N + i] = (int)m;
    }
    if (bad) atomicOr(status, ST_INTERNAL);
    if (last && s) atomicAdd((u64 *)&count[i], (u64)s);
}

// one thread per sorted row: med[r], mad[r] as np.median and np.median(np.abs(y - med))
__global__ void __launch_bounds__(MM_THREADS) medmad_kernel(const double *__restrict__ sorted, const i64 R,
                                                            const i64 n, double *__restrict__ med,
                                                            double *__restrict__ mad) {
    const i64 r = (i64)blockIdx.x * MM_THREADS + threadIdx.x;
    if (r >= R) return;
    const PlainRow s{sorted + r * n};
    const double md = row_median(s, n), v = row_mad(s, n, md);
    med[r] = md;
    mad[r] = v;
}

// grid (point tiles, time tiles of tpt time points).  Y rows r = tt * kb + kk (leading dimension ldY), med / mad
// [tb * kb].
// out [tb][N] after the last direction block, else the running max run [tb][N].
__global__ void __launch_bounds__(RD_THREADS) pd_max_kernel(const double *__restrict__ Y, const i64 ldY,
                                                            const double *__restrict__ med,
                                                            const double *__restrict__ mad, const i64 N,
                                                            const i64 kb, const i64 tb, const i64 tpt,
                                                            double *__restrict__ run, const int first,
                                                            double *__restrict__ out) {
    const i64 i = (i64)blockIdx.x * RD_THREADS + threadIdx.x;
    if (i >= N) return;
    const i64 t0 = (i64)blockIdx.y * tpt;
    const i64 t1 = t0 + tpt < tb ? t0 + tpt : tb;
    for (i64 t = t0; t < t1; ++t) {
        u64 m = first ? 0ull : (u64)__double_as_longlong(run[t * N + i]);
        for (i64 kk = 0; kk < kb; ++kk) {
            const i64 r = t * kb + kk;
            const double y = Y[r * ldY + i], md = med[r], s = mad[r];
            const u64 ob = (u64)__double_as_longlong(outlyingness(y, md, s));
            m = ob > m ? ob : m;
        }
        (out ? out : run)[t * N + i] = __longlong_as_double((long long)m);
    }
}

i64 projection_rows_max(i64 N) {
    const i64 rows = (i64)(PJ_BUDGET / ((size_t)(N + (N & 1)) * sizeof(double)));
    return rows < 1 ? 1 : rows;
}

void projection_blocks(i64 rows_max, i64 T, i64 K, i64 *kb_max, i64 *tb_max) {
    // a time block keeps all K directions when K rows fit
    i64 kb = K <= rows_max ? K : rows_max;
    if (kb > PJ_MAX_KB) kb = PJ_MAX_KB;
    i64 tb = kb == K ? rows_max / K : 1;
    if (tb > T) tb = T;
    if (tb > PJ_MAX_TB) tb = PJ_MAX_TB;
    *kb_max = kb;
    *tb_max = tb;
}

int project_device(sd_ctx *ctx, const double *dF, i64 N, i64 T, int d, const double *dU, i64 kb, i64 t0, i64 tb,
                   double *Y, i64 ldY) {
    const int TT = d <= PJ_W ? PJ_W / d : 1;
    const dim3 pgrid((unsigned)ceil_div(N, PJ_PTS), (unsigned)ceil_div(kb, PJ_DIRS), (unsigned)ceil_div(tb, TT));
    projection_kernel<<<pgrid, PJ_THREADS, 0, ctx->stream>>>(dF, N, T, d, dU, kb, t0, tb, TT, Y, ldY);
    ctx->last.launches++;
    SD_CUDA(cudaGetLastError());
    return SD_OK;
}

int projection_device(sd_ctx *ctx, const double *dF, i64 N, i64 T, int d, i64 ldX, const double *dU, i64 K,
                      ProjKind kind, i64 *d_count, double *d_o, double *med_out, double *mad_out,
                      cudaMemcpyKind out_kind) {
    if (N < 1 || T < 1 || K < 1 || (dU ? d < 1 : (K != 1 || ldX < N))) {
        set_error("projection depth: bad shape N=%lld T=%lld d=%d K=%lld", (long long)N, (long long)T, d,
                  (long long)K);
        return SD_ERR_INVALID;
    }
    if (N >= (1ll << 31)) {
        set_error("projection depth: N=%lld exceeds 2^31-1", (long long)N);
        return SD_ERR_UNSUPPORTED;
    }
    cudaStream_t st = ctx->stream;
    const bool rt = kind == PJ_TUKEY;
    if (dU) SD_TRY(finite_check_device(ctx, dF, 1, N * T * d, N * T * d));
    else SD_TRY(finite_check_device(ctx, dF, T, N, ldX));
    const i64 ldY = dU ? N + (N & 1) : ldX;
    i64 rows_max = projection_rows_max(N);
    int *rb = nullptr, *ra = nullptr;
    if (rt) {
        i64 RB = 0;
        SD_TRY(rank_block_workspace(ctx, rows_max < T * K ? rows_max : T * K, 2 * N, &RB, &rb));
        if (rows_max > RB) rows_max = RB;
    }
    i64 kb_max, tb_max;
    projection_blocks(rows_max, T, K, &kb_max, &tb_max);
    const i64 R = tb_max * kb_max;
    if (rt) ra = rb + (size_t)R * N;
    double *Y = nullptr;
    if (dU) {
        SD_TRY(ctx->buf[BUF_PROJ].reserve((size_t)R * ldY * sizeof(double)));
        Y = ctx->buf[BUF_PROJ].as<double>();
    }
    double *sorted = nullptr;
    if (!rt) {
        SD_TRY(ctx->buf[BUF_PSORT].reserve((size_t)R * N * sizeof(double)));
        sorted = ctx->buf[BUF_PSORT].as<double>();
    }
    const bool split = kb_max < K;  // direction blocks continue a running value
    SD_TRY(ctx->buf[BUF_PRED].reserve(((split ? (size_t)tb_max * N : 0) + (rt ? 0 : 2 * (size_t)R) + 1) *
                                      sizeof(double)));
    double *pred = ctx->buf[BUF_PRED].as<double>();
    double *d_med = pred + (split ? (size_t)tb_max * N : 0), *d_mad = d_med + R;
    if (rt) SD_CUDA(cudaMemsetAsync(d_count, 0, (size_t)N * sizeof(i64), st));
    for (i64 t0 = 0; t0 < T; t0 += tb_max) {
        const i64 tb = T - t0 < tb_max ? T - t0 : tb_max;
        // time points per reduction thread: up to RD_MAX_ROWS while N tb / tpt threads still fill ~2 occupancies
        i64 tpt = N * tb / (2 * 2048 * (i64)ctx->sm_count);
        if (tpt > RD_MAX_ROWS) tpt = RD_MAX_ROWS;
        if (tpt < 1) tpt = 1;
        const dim3 rgrid((unsigned)ceil_div(N, RD_THREADS), (unsigned)ceil_div(tb, tpt));
        for (i64 k0 = 0; k0 < K; k0 += kb_max) {
            const i64 kb = K - k0 < kb_max ? K - k0 : kb_max;
            const i64 rows = tb * kb;
            const double *Yb = dF + t0 * ldX;
            if (dU) {
                SD_TRY(project_device(ctx, dF, N, T, d, dU + k0 * d, kb, t0, tb, Y, ldY));
                Yb = Y;
            }
            const int first = k0 == 0, last = k0 + kb == K;
            if (rt) {
                SD_TRY(rank_rows_device(ctx, Yb, rows, N, ldY, rb, ra));
                rt_min_kernel<<<rgrid, RD_THREADS, 0, st>>>(rb, ra, N, kb, tb, tpt, (int *)pred, first, last, d_count,
                                                            ctx->d_status);
                ctx->last.launches++;
                SD_CUDA(cudaGetLastError());
                continue;
            }
            SD_TRY(sort_rows_device(ctx, Yb, rows, N, ldY, sorted));
            medmad_kernel<<<(unsigned)ceil_div(rows, MM_THREADS), MM_THREADS, 0, st>>>(sorted, rows, N, d_med, d_mad);
            pd_max_kernel<<<rgrid, RD_THREADS, 0, st>>>(Yb, ldY, d_med, d_mad, N, kb, tb, tpt, pred, first,
                                                        last ? d_o + t0 * N : nullptr);
            ctx->last.launches += 2;
            SD_CUDA(cudaGetLastError());
            // rows (tt, kk) of the block are entries (t0 + tt, k0 + kk) of the [T, K] outputs
            if (med_out)
                SD_CUDA(cudaMemcpy2DAsync(med_out + t0 * K + k0, (size_t)K * sizeof(double), d_med,
                                          (size_t)kb * sizeof(double), (size_t)kb * sizeof(double), (size_t)tb,
                                          out_kind, st));
            if (mad_out)
                SD_CUDA(cudaMemcpy2DAsync(mad_out + t0 * K + k0, (size_t)K * sizeof(double), d_mad,
                                          (size_t)kb * sizeof(double), (size_t)kb * sizeof(double), (size_t)tb,
                                          out_kind, st));
        }
    }
    return SD_OK;
}

}  // namespace sd
