// reference_proj.cu -- fitted references for random projection depths (K13): a reference sample's projections sorted
// once on the device, new observations scored against them by binary search.
//
// Out-of-sample convention (as K7 / K9): a new observation g gets exactly the depth the in-sample call (K12) gives it
// after g alone is appended to the reference S, with the same directions U.  Per row (t, k), with s the sorted
// projections of S (nS values), y = g's projection, b / a = #s strictly below / above y:
//   random Tukey:  h = (nS + 1) - max(b, a);  count(g) = sum_t min_k h   (rt_min_kernel's formula with N = nS + 1)
//   projection:    med' / MAD' of the virtual sorted row v = s with y inserted at p = b (InsertedRow, never written),
//                  selected by row_median / row_mad exactly as medmad_kernel selects them on a real row (sorted_row.cuh), and
//                  O(g, t) = max_k |y - med'| / MAD'.
// So the counts and the bits of O are those of the in-sample call on S + [g] by construction.
//
// Build (projection_sort_rows_device): index[(t * K + k) * nS + j] = the j-th smallest of y_k(., t) over S.  Blocked
// like projection_device: projection_kernel writes a block of rows into BUF_PROJ within PJ_BUDGET, sort_rows_device
// (K9) sorts them straight into the caller's index slice.  A block (t0 .. t0 + tb, k0 .. k0 + kb) is kb == K or
// tb == 1, so its rows are consecutive rows (t0 * K + k0 ..) of the index.  A projection that overflows is caught by
// the rank pass's finite check (SD_ERR_NONFINITE), as in-sample.  Univariate curves use K9's index (K = 1, y = x).
//
// Query (projection_sorted_device): the new curves are finite-checked, projected in blocks as above (ldY = nY rounded
// up to even) and then one of
//   sorted_tukey_kernel        thread (g, up to 32 time points): per (t, k) the paired bound search and h, a running
//                              int32 min; across direction blocks through BUF_PRED; after the last one a single int64
//                              atomic of sum_t.
//   sorted_outlyingness_kernel same grid: per (t, k) the lower bound p, med' / MAD' on the virtual row and O, a
//                              running max compared as u64 bit patterns (as pd_max_kernel); O[t][g] after the last
//                              direction block.
// Y is read coalesced along g.  Fewer time points per thread when n_Y * tb / 32 threads would not fill ~2 occupancies
// (as rt_min_kernel / sorted_terms_kernel).  No rank pass runs on the new projections, so the kernels flag a
// non-finite one themselves (ST_NONFINITE -> SD_ERR_NONFINITE: the pooled in-sample call refuses the same inputs).
// b, a outside 0 <= b, a, b + a <= nS sets ST_INTERNAL (never a trap); every index read stays in [0, nS).
#include "sorted_row.cuh"

namespace sd {

constexpr int SQ_THREADS = 256;
constexpr i64 SQ_MAX_ROWS = 32;  // time points per thread when there are enough (t, g) pairs

// grid (new-curve tiles, time tiles of tpt time points).  Block rows r = tt * kb + kk: Y[r * ldY + g], index row
// (tt * K + kk) * nS.  run [tb][nY] while direction blocks continue.
__global__ void __launch_bounds__(SQ_THREADS) sorted_tukey_kernel(const double *__restrict__ index, const i64 nS,
                                                                  const i64 K, const double *__restrict__ Y,
                                                                  const i64 ldY, const i64 nY, const i64 kb,
                                                                  const i64 tb, const i64 tpt, int *__restrict__ run,
                                                                  const int first, const int last,
                                                                  i64 *__restrict__ count, int *__restrict__ status) {
    const i64 g = (i64)blockIdx.x * SQ_THREADS + threadIdx.x;
    if (g >= nY) return;
    const i64 t0 = (i64)blockIdx.y * tpt;
    const i64 t1 = t0 + tpt < tb ? t0 + tpt : tb;
    i64 s = 0;
    bool bad = false, nonfinite = false;
    for (i64 t = t0; t < t1; ++t) {
        i64 m = first ? nS + 1 : run[t * nY + g];
        for (i64 kk = 0; kk < kb; ++kk) {
            const double y = Y[(t * kb + kk) * ldY + g];
            nonfinite |= !isfinite(y);
            i64 b, a;
            sorted_bounds(index + (t * K + kk) * nS, nS, y, b, a);
            if (b < 0 || a < 0 || b + a > nS) {
                bad = true;
                continue;
            }
            const i64 h = nS + 1 - (b > a ? b : a);
            m = h < m ? h : m;
        }
        if (last) s += m;
        else run[t * nY + g] = (int)m;
    }
    if (bad) atomicOr(status, ST_INTERNAL);
    if (nonfinite) atomicOr(status, ST_NONFINITE);
    if (last && s) atomicAdd((u64 *)&count[g], (u64)s);
}

// same grid and rows; out [tb][nY] after the last direction block, else the running max run [tb][nY]
__global__ void __launch_bounds__(SQ_THREADS) sorted_outlyingness_kernel(
    const double *__restrict__ index, const i64 nS, const i64 K, const double *__restrict__ Y, const i64 ldY,
    const i64 nY, const i64 kb, const i64 tb, const i64 tpt, double *__restrict__ run, const int first,
    double *__restrict__ out, int *__restrict__ status) {
    const i64 g = (i64)blockIdx.x * SQ_THREADS + threadIdx.x;
    if (g >= nY) return;
    const i64 t0 = (i64)blockIdx.y * tpt;
    const i64 t1 = t0 + tpt < tb ? t0 + tpt : tb;
    bool bad = false, nonfinite = false;
    for (i64 t = t0; t < t1; ++t) {
        u64 m = first ? 0ull : (u64)__double_as_longlong(run[t * nY + g]);
        for (i64 kk = 0; kk < kb; ++kk) {
            const double y = Y[(t * kb + kk) * ldY + g];
            nonfinite |= !isfinite(y);
            const double *row = index + (t * K + kk) * nS;
            i64 b, a;
            sorted_bounds(row, nS, y, b, a);  // only b is used: the upper-bound chain is dead code
            if (b < 0 || b > nS) {
                bad = true;
                continue;
            }
            const InsertedRow v{row, b, y};
            const double md = row_median(v, nS + 1);
            const u64 ob = (u64)__double_as_longlong(outlyingness(y, md, row_mad(v, nS + 1, md)));
            m = ob > m ? ob : m;
        }
        (out ? out : run)[t * nY + g] = __longlong_as_double((long long)m);
    }
    if (bad) atomicOr(status, ST_INTERNAL);
    if (nonfinite) atomicOr(status, ST_NONFINITE);
}

int projection_sort_rows_device(sd_ctx *ctx, const double *dF, i64 nS, i64 T, int d, const double *dU, i64 K,
                                double *d_sorted) {
    if (nS < 1 || T < 1 || d < 1 || K < 1 || !dU) {
        set_error("projected reference: bad shape nS=%lld T=%lld d=%d K=%lld", (long long)nS, (long long)T, d,
                  (long long)K);
        return SD_ERR_INVALID;
    }
    if (nS >= (1ll << 31)) {
        set_error("projected reference: nS=%lld exceeds 2^31-1", (long long)nS);
        return SD_ERR_UNSUPPORTED;
    }
    SD_TRY(finite_check_device(ctx, dF, 1, nS * T * d, nS * T * d));
    const i64 ldY = nS + (nS & 1);
    i64 kb_max, tb_max;
    projection_blocks(projection_rows_max(nS), T, K, &kb_max, &tb_max);
    SD_TRY(ctx->buf[BUF_PROJ].reserve((size_t)tb_max * kb_max * ldY * sizeof(double)));
    double *Y = ctx->buf[BUF_PROJ].as<double>();
    for (i64 t0 = 0; t0 < T; t0 += tb_max) {
        const i64 tb = T - t0 < tb_max ? T - t0 : tb_max;
        for (i64 k0 = 0; k0 < K; k0 += kb_max) {
            const i64 kb = K - k0 < kb_max ? K - k0 : kb_max;
            SD_TRY(project_device(ctx, dF, nS, T, d, dU + k0 * d, kb, t0, tb, Y, ldY));
            SD_TRY(sort_rows_device(ctx, Y, tb * kb, nS, ldY, d_sorted + (t0 * K + k0) * nS));
        }
    }
    return SD_OK;
}

int projection_sorted_device(sd_ctx *ctx, const double *d_sorted, i64 nS, i64 T, const double *dY, i64 nY, i64 ldY,
                             int d, const double *dU, i64 K, ProjKind kind, i64 *d_count, double *d_o) {
    if (nS < 1 || T < 1 || nY < 0 || K < 1 || (dU ? d < 1 : (K != 1 || ldY < nY))) {
        set_error("projected reference query: bad shape nS=%lld T=%lld nY=%lld d=%d K=%lld", (long long)nS,
                  (long long)T, (long long)nY, d, (long long)K);
        return SD_ERR_INVALID;
    }
    if (nS + 1 >= (1ll << 31)) {
        set_error("projected reference query: nS + 1 = %lld exceeds 2^31-1", (long long)(nS + 1));
        return SD_ERR_UNSUPPORTED;
    }
    if (nY == 0) return SD_OK;
    cudaStream_t st = ctx->stream;
    const bool rt = kind == PJ_TUKEY;
    if (dU) SD_TRY(finite_check_device(ctx, dY, 1, nY * T * d, nY * T * d));
    else SD_TRY(finite_check_device(ctx, dY, T, nY, ldY));
    const i64 ldP = dU ? nY + (nY & 1) : ldY;
    i64 kb_max, tb_max;
    projection_blocks(projection_rows_max(nY), T, K, &kb_max, &tb_max);
    double *P = nullptr;
    if (dU) {
        SD_TRY(ctx->buf[BUF_PROJ].reserve((size_t)tb_max * kb_max * ldP * sizeof(double)));
        P = ctx->buf[BUF_PROJ].as<double>();
    }
    const bool split = kb_max < K;  // direction blocks continue a running value
    SD_TRY(ctx->buf[BUF_PRED].reserve(((split ? (size_t)tb_max * nY : 0) + 1) * sizeof(double)));
    double *pred = ctx->buf[BUF_PRED].as<double>();
    if (rt) SD_CUDA(cudaMemsetAsync(d_count, 0, (size_t)nY * sizeof(i64), st));
    for (i64 t0 = 0; t0 < T; t0 += tb_max) {
        const i64 tb = T - t0 < tb_max ? T - t0 : tb_max;
        i64 tpt = nY * tb / (2 * 2048 * (i64)ctx->sm_count);  // ~2 full occupancies
        if (tpt > SQ_MAX_ROWS) tpt = SQ_MAX_ROWS;
        if (tpt < 1) tpt = 1;
        const dim3 grid((unsigned)ceil_div(nY, SQ_THREADS), (unsigned)ceil_div(tb, tpt));
        for (i64 k0 = 0; k0 < K; k0 += kb_max) {
            const i64 kb = K - k0 < kb_max ? K - k0 : kb_max;
            const double *Yb = dY + t0 * ldY;
            if (dU) {
                SD_TRY(project_device(ctx, dY, nY, T, d, dU + k0 * d, kb, t0, tb, P, ldP));
                Yb = P;
            }
            const double *ib = d_sorted + (t0 * K + k0) * nS;
            const int first = k0 == 0, last = k0 + kb == K;
            if (rt)
                sorted_tukey_kernel<<<grid, SQ_THREADS, 0, st>>>(ib, nS, K, Yb, ldP, nY, kb, tb, tpt, (int *)pred,
                                                                 first, last, d_count, ctx->d_status);
            else
                sorted_outlyingness_kernel<<<grid, SQ_THREADS, 0, st>>>(ib, nS, K, Yb, ldP, nY, kb, tb, tpt, pred,
                                                                        first, last ? d_o + t0 * nY : nullptr,
                                                                        ctx->d_status);
            ctx->last.launches++;
            SD_CUDA(cudaGetLastError());
        }
    }
    return SD_OK;
}

}  // namespace sd
