// api.cu -- the extern "C" entry points of include/statdepth_b200.h.  Host-buffer entry points copy their inputs to
// the device, run the kernels and copy the results back; the _dev variants take device pointers.
//
// Adding an entry point: check the arguments that need neither the context nor the device (sizes, layout, required
// buffers), then return call(...) with two lambdas.  `stage` uploads the host inputs, reserves the workspace the
// results land in and registers their copies back (Staging); `run` queues the device work.  call() checks the
// context and the main input / output pointers, turns any C++ exception into SD_ERR_INVALID, and brackets the body
// with begin_call / mark / end_call, so that h2d_ns, kernel_ns and d2h_ns mean the same in every entry point.  A
// host / _dev pair shares one static body that takes a `dev` flag: the checks and the device work are written once,
// and the host side alone stages.  Checks only the host can make (query, pool and member ids in range) stay in its
// `stage`.
#include <thread>
#include <vector>

#include "common.cuh"

namespace sd {

// strict J = 2 by enumeration: bit kernel, or the dense Gram when a probe of 8 queries shows that the bit
// kernel would drown in survivors (non-crossing / tie-heavy curves)
static int strict_enumerate(sd_ctx *ctx, const double *dX, i64 T, i64 n, i64 ld, const i64 *d_q, i64 nq, i64 *d_out) {
    if (ctx->bd_impl == SD_BD_GEMM) {
        ctx->last.bd_impl_used = SD_BD_GEMM;
        return bd_strict_gemm_device(ctx, dX, T, n, ld, d_q, nq, d_out);
    }
    if (ctx->last.bd_impl_used == 0) ctx->last.bd_impl_used = SD_BD_BITS;
    constexpr i64 PROBE = 8;
    if (ctx->bd_impl == SD_BD_BITS || nq <= 4 * PROBE || n < 1024)
        return bd_strict_device(ctx, dX, T, n, ld, d_q, nq, 2, d_out);
    SD_TRY(ctx->buf[BUF_WORK].reserve(sizeof(u64)));
    u64 *d_hits = ctx->buf[BUF_WORK].as<u64>();
    SD_CUDA(cudaMemsetAsync(d_hits, 0, sizeof(u64), ctx->stream));
    SD_TRY(bd_strict_device(ctx, dX, T, n, ld, d_q, PROBE, 2, d_out, d_hits));
    u64 h_hits = 0;
    SD_CUDA(cudaMemcpyAsync(&h_hits, d_hits, sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream));
    SD_CUDA(cudaStreamSynchronize(ctx->stream));
    const double pairs = (double)PROBE * 0.5 * (double)(n - 1) * (double)(n - 2);
    if ((double)h_hits > 0.02 * pairs) {
        ctx->last.bd_impl_used = SD_BD_GEMM;
        return bd_strict_gemm_device(ctx, dX, T, n, ld, d_q + PROBE, nq - PROBE, d_out + PROBE);
    }
    ctx->last.bd_impl_used = SD_BD_BITS;
    return bd_strict_device(ctx, dX, T, n, ld, d_q + PROBE, nq - PROBE, 2, d_out + PROBE);
}

bool relaxed_overflows(i64 T, i64 others, int j) {
    const long double full = (j == 2) ? (long double)others * (others - 1) / 2.0L
                                      : (long double)others * (others - 1) * (others - 2) / 6.0L;
    // j = 3: the kernels form 3 * C(m, 3) before dividing (comb3_dev), so that intermediate must fit as well
    return full * (long double)T >= 9.0e18L || (j == 3 && 3.0L * full >= 9.0e18L);
}

int relaxed_overflow_check(i64 T, i64 others, int j, const char *who) {
    if (!relaxed_overflows(T, others, j)) return SD_OK;
    set_error("%s: T*C(%lld,%d) overflows int64 for T=%lld", who, (long long)others, j, (long long)T);
    return SD_ERR_OVERFLOW;
}

// dispatch one subset size j on device-resident data
int band_depth_device(sd_ctx *ctx, const double *dX, i64 T, i64 n, i64 ld, const i64 *d_q, i64 nq, int j,
                      int relax, i64 *d_out) {
    if (j != 2 && j != 3) {
        set_error("band depth: subset size j=%d not supported on the device (2 or 3)", j);
        return SD_ERR_UNSUPPORTED;
    }
    if (!relax) {
        if (!d_q) {  // all curves: the strict drivers take an explicit list (the probe and the chunks offset it)
            SD_TRY(ctx->buf[BUF_QIDX].reserve((size_t)nq * sizeof(i64)));
            i64 *q = ctx->buf[BUF_QIDX].as<i64>();
            SD_TRY(iota_from_device(ctx, q, nq, 0));
            d_q = q;
        }
        if (j == 3) {
            ctx->last.bd_impl_used = SD_BD_BITS;
            return bd_strict_device(ctx, dX, T, n, ld, d_q, nq, 3, d_out);
        }
        ctx->last.bd_impl_used = 0;
        const bool match = (ctx->bd_impl == SD_BD_MATCH || ctx->bd_impl == SD_BD_AUTO) && bd_match_supported(T, n);
        if (!match) return strict_enumerate(ctx, dX, T, n, ld, d_q, nq, d_out);
        i64 nfb = 0;
        SD_TRY(bd_strict_match_device(ctx, dX, T, n, ld, d_q, nq, d_out, strict_enumerate, &nfb));
        if (2 * nfb <= nq) ctx->last.bd_impl_used = SD_BD_MATCH;  // else: what strict_enumerate chose
        return SD_OK;
    }
    SD_TRY(relaxed_overflow_check(T, n - 1, j, "band depth"));
    SD_TRY(ctx->buf[BUF_ACC].reserve((size_t)n * 2 * sizeof(i64)));
    i64 *acc2 = ctx->buf[BUF_ACC].as<i64>();
    i64 *acc3 = acc2 + n;
    if (!d_q && j == 2)  // all curves, in order: the finish kernel writes the caller's buffer, no gather launch
        return mbd_all_device(ctx, dX, T, n, ld, d_out, nullptr);
    SD_TRY(mbd_all_device(ctx, dX, T, n, ld, acc2, j == 3 ? acc3 : nullptr));
    return gather_i64_device(ctx, j == 2 ? acc2 : acc3, d_q, nq, d_out);
}

static int check_common(sd_ctx *ctx, const void *in, const void *out, const char *who) {
    if (!ctx) {
        set_error("%s: NULL context", who);
        return SD_ERR_INVALID;
    }
    if (!in || !out) {
        set_error("%s: NULL buffer", who);
        return SD_ERR_INVALID;
    }
    return SD_OK;
}

static int check_matrix(const char *who, i64 T, i64 n, i64 ld, int layout) {
    SD_REQUIRE(T >= 1 && n >= 1, "%s: bad sizes T=%lld n=%lld", who, (long long)T, (long long)n);
    SD_REQUIRE(layout == SD_LAYOUT_TN || layout == SD_LAYOUT_NT, "%s: bad layout %d", who, layout);
    SD_REQUIRE(ld >= (layout == SD_LAYOUT_TN ? n : T), "%s: ld=%lld too small", who, (long long)ld);
    return SD_OK;
}

// upload helper: host matrix [rows, cols] with leading dimension ld -> dense device [rows, cols]
static int upload_matrix(sd_ctx *ctx, int slot, const double *h, i64 rows, i64 cols, i64 ld, double **d) {
    SD_TRY(ctx->buf[slot].reserve((size_t)(rows * cols > 0 ? rows * cols : 1) * sizeof(double)));
    *d = ctx->buf[slot].as<double>();
    if (rows == 0 || cols == 0) return SD_OK;
    if (ld == cols || rows == 1) {
        SD_CUDA(cudaMemcpyAsync(*d, h, (size_t)rows * cols * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    } else {
        SD_CUDA(cudaMemcpy2DAsync(*d, (size_t)cols * sizeof(double), h, (size_t)ld * sizeof(double),
                                  (size_t)cols * sizeof(double), (size_t)rows, cudaMemcpyHostToDevice,
                                  ctx->stream));
    }
    return SD_OK;
}

static int upload_queries(sd_ctx *ctx, const int64_t *h_q, i64 nq, i64 n, const i64 **d_q, const char *who) {
    *d_q = nullptr;
    if (!h_q) {
        if (nq != n) {
            set_error("%s: query_idx == NULL requires nq == n", who);
            return SD_ERR_INVALID;
        }
        return SD_OK;
    }
    for (i64 i = 0; i < nq; ++i)
        if (h_q[i] < 0 || h_q[i] >= n) {
            set_error("%s: query_idx[%lld]=%lld out of range [0,%lld)", who, (long long)i, (long long)h_q[i],
                      (long long)n);
            return SD_ERR_INVALID;
        }
    SD_TRY(ctx->buf[BUF_MISC].reserve((size_t)(nq > 0 ? nq : 1) * sizeof(i64)));
    i64 *dq = ctx->buf[BUF_MISC].as<i64>();
    if (nq > 0)
        SD_CUDA(cudaMemcpyAsync(dq, h_q, (size_t)nq * sizeof(i64), cudaMemcpyHostToDevice, ctx->stream));
    *d_q = dq;
    return SD_OK;
}

// What a host-buffer call does besides its kernels: the transpose of an SD_LAYOUT_NT upload, run once the kernel
// phase has begun (so it counts in kernel_ns), and the copies of the results back to the caller, queued after it.
struct Staging {
    sd_ctx *ctx;
    const double *nt = nullptr;  // uploaded [nt_rows, nt_cols], transposed into nt_out
    double *nt_out = nullptr;
    i64 nt_rows = 0, nt_cols = 0;
    bool h2d_overlapped = false;  // the upload runs inside the kernel phase (band_depth_pipelined): h2d_ns is 0
    struct Copy {
        void *host;
        const void *dev;
        size_t bytes;
    };
    std::vector<Copy> down;

    // a result copied back after the kernels; an optional output the caller passed as NULL is skipped
    void download(void *host, const void *dev, size_t bytes) { down.push_back({host, dev, bytes}); }

    // count results in workspace slot `slot`, copied back to host
    template <class V>
    int output(int slot, void *host, i64 count, V **dev) {
        SD_TRY(ctx->buf[slot].reserve((size_t)(count > 0 ? count : 1) * sizeof(V)));
        *dev = ctx->buf[slot].as<V>();
        download(host, *dev, (size_t)count * sizeof(V));
        return SD_OK;
    }

    // host matrix in either layout -> dense device [T, n] in BUF_IN (SD_LAYOUT_NT goes to BUF_IN2 first)
    int upload_tn(const double *X, i64 T, i64 n, i64 ld, int layout, const double **dX) {
        double *d = nullptr;
        if (layout == SD_LAYOUT_TN) {
            SD_TRY(upload_matrix(ctx, BUF_IN, X, T, n, ld, &d));
        } else {
            SD_TRY(upload_matrix(ctx, BUF_IN2, X, n, T, ld, &d));
            nt = d;
            nt_rows = n;
            nt_cols = T;
            SD_TRY(ctx->buf[BUF_IN].reserve((size_t)T * n * sizeof(double)));
            d = nt_out = ctx->buf[BUF_IN].as<double>();
        }
        *dX = d;
        return SD_OK;
    }
};

static int no_stage(Staging &) { return SD_OK; }

// The one call path of every entry point: stage (uploads, before mark 1), run (the device work, between marks 1 and
// 2), then the copies back.  `host`: the call copies to or from host buffers (end_call times h2d and d2h).
// `may_defer`: under SD_OPT_ASYNC_DEVICE the call stays open on ctx->stream and sd_sync() completes it.
template <class Stage, class Run>
static int call(sd_ctx *ctx, const char *who, const void *in, const void *out, bool host, Stage stage, Run run,
                bool may_defer = false) {
    SD_TRY(check_common(ctx, in, out, who));
    try {
        Staging s{ctx};
        SD_TRY(begin_call(ctx));
        SD_TRY(stage(s));
        SD_TRY(mark(ctx, 1));
        if (s.nt) SD_TRY(transpose_device(ctx, s.nt, s.nt_rows, s.nt_cols, s.nt_cols, s.nt_out));
        SD_TRY(run());
        SD_TRY(mark(ctx, 2));
        for (const Staging::Copy &c : s.down)
            if (c.host && c.bytes > 0)
                SD_CUDA(cudaMemcpyAsync(c.host, c.dev, c.bytes, cudaMemcpyDeviceToHost, ctx->stream));
        if (may_defer && ctx->async_device) {
            ctx->pending = 1;
            return SD_OK;
        }
        const int st = end_call(ctx, host);
        if (s.h2d_overlapped) ctx->last.h2d_ns = 0;
        return st;
    } catch (...) {  // std::bad_alloc from host-side staging (vectors, threads): the ABI never throws
        set_error("%s: out of host memory", who);
        return SD_ERR_INVALID;
    }
}

// Pageable host input (what FunctionalDepth([DataFrame]) hands over): cudaMemcpyAsync from unregistered memory is a
// synchronous, single-threaded staged copy (~11 GB/s measured: 74 ms for the 819 MB of config 2 against 15 ms from
// pinned memory).  The blocks are instead copied into two pinned staging buffers by a few host threads while the
// previous block's DMA and ranking run.
static bool host_is_pageable(const void *p) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return true;
    }
    return a.type == cudaMemoryTypeUnregistered;
}

static void parallel_copy_rows(double *dst, const double *src, i64 rows, i64 n, i64 ld, int nthreads) {
    if (nthreads < 1) nthreads = 1;
    std::vector<std::thread> th;
    const i64 per = ceil_div(rows, nthreads);
    for (int t = 0; t < nthreads; ++t) {
        const i64 r0 = t * per, r1 = r0 + per < rows ? r0 + per : rows;
        if (r0 >= r1) break;
        th.emplace_back([=]() {
            if (ld == n) memcpy(dst + r0 * n, src + r0 * ld, (size_t)(r1 - r0) * n * sizeof(double));
            else
                for (i64 r = r0; r < r1; ++r) memcpy(dst + r * n, src + r * ld, (size_t)n * sizeof(double));
        });
    }
    for (auto &t : th) t.join();
}

// Relaxed band depth of a host matrix, streamed in row blocks (see sd_band_depth_f64).  Timings: h2d_ns is 0
// and kernel_ns covers the overlapped copy + ranking region.
static int band_depth_pipelined(sd_ctx *ctx, const double *X, i64 T, i64 n, i64 ld, const int64_t *query_idx, i64 nq,
                                int j, int64_t *count_out, const char *who) {
    i64 RB = ceil_div(T, 8);                       // 8 blocks ...
    const i64 min_rows = ceil_div((i64)(32u << 20), n * (i64)sizeof(double));
    if (RB < min_rows) RB = min_rows;              // ... of at least 32 MB
    if (RB > T) RB = T;
    double *dbuf[2] = {nullptr, nullptr};
    const i64 *d_q = nullptr;
    i64 *d_out = nullptr, *acc2 = nullptr, *acc3 = nullptr;
    const auto stage = [&](Staging &s) -> int {
        SD_TRY(relaxed_overflow_check(T, n - 1, j, "band depth"));
        SD_TRY(ctx->buf[BUF_IN].reserve((size_t)2 * RB * n * sizeof(double)));
        dbuf[0] = ctx->buf[BUF_IN].as<double>();
        dbuf[1] = dbuf[0] + (size_t)RB * n;
        SD_TRY(upload_queries(ctx, query_idx, nq, n, &d_q, who));
        SD_TRY(s.output(BUF_OUT, count_out, nq, &d_out));
        SD_TRY(ctx->buf[BUF_ACC].reserve((size_t)n * 2 * sizeof(i64)));
        acc2 = ctx->buf[BUF_ACC].as<i64>();
        acc3 = acc2 + n;
        s.h2d_overlapped = true;
        return SD_OK;
    };
    const auto run = [&]() -> int {
        // the copy stream must not overtake work already queued on the main stream (query upload, status reset)
        SD_CUDA(cudaEventRecord(ctx->ev_pipe[2], ctx->stream));
        SD_CUDA(cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_pipe[2], 0));
        const bool staged = host_is_pageable(X);
        int nthreads = (int)std::thread::hardware_concurrency();
        if (nthreads > 8) nthreads = 8;
        if (staged) {
            for (int s = 0; s < 2; ++s) {
                if (ctx->stage_cap[s] < (size_t)RB * n * sizeof(double)) {
                    if (ctx->stage[s]) cudaFreeHost(ctx->stage[s]);
                    ctx->stage[s] = nullptr;
                    ctx->stage_cap[s] = 0;
                    SD_CUDA(cudaHostAlloc(&ctx->stage[s], (size_t)RB * n * sizeof(double), cudaHostAllocDefault));
                    ctx->stage_cap[s] = (size_t)RB * n * sizeof(double);
                }
                if (!ctx->ev_stage[s]) SD_CUDA(cudaEventCreateWithFlags(&ctx->ev_stage[s], cudaEventDisableTiming));
            }
        }
        // an error inside the loop must not return while a copy out of the caller's buffer is still in flight
        ctx->mbd_no_wait = 1;  // the host must keep feeding the copy stream while earlier blocks are ranked
        const int loop_status = [&]() -> int {
            int k = 0;
            for (i64 r0 = 0; r0 < T; r0 += RB, ++k) {
                const int s = k & 1;
                const i64 rows = T - r0 < RB ? T - r0 : RB;
                if (k >= 2) SD_CUDA(cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_pipe[2 + s], 0));  // k-2 consumed
                if (staged) {
                    if (k >= 2) SD_CUDA(cudaEventSynchronize(ctx->ev_stage[s]));  // the DMA out of this buffer is done
                    parallel_copy_rows((double *)ctx->stage[s], X + r0 * ld, rows, n, ld, nthreads);
                    SD_CUDA(cudaMemcpyAsync(dbuf[s], ctx->stage[s], (size_t)rows * n * sizeof(double),
                                            cudaMemcpyHostToDevice, ctx->copy_stream));
                    SD_CUDA(cudaEventRecord(ctx->ev_stage[s], ctx->copy_stream));
                } else if (ld == n) {
                    SD_CUDA(cudaMemcpyAsync(dbuf[s], X + r0 * ld, (size_t)rows * n * sizeof(double),
                                            cudaMemcpyHostToDevice, ctx->copy_stream));
                } else {
                    SD_CUDA(cudaMemcpy2DAsync(dbuf[s], (size_t)n * sizeof(double), X + r0 * ld,
                                              (size_t)ld * sizeof(double), (size_t)n * sizeof(double), (size_t)rows,
                                              cudaMemcpyHostToDevice, ctx->copy_stream));
                }
                SD_CUDA(cudaEventRecord(ctx->ev_pipe[s], ctx->copy_stream));
                SD_CUDA(cudaStreamWaitEvent(ctx->stream, ctx->ev_pipe[s], 0));
                SD_TRY(mbd_all_device(ctx, dbuf[s], rows, n, n, acc2, j == 3 ? acc3 : nullptr, k > 0));
                SD_CUDA(cudaEventRecord(ctx->ev_pipe[2 + s], ctx->stream));
            }
            return SD_OK;
        }();
        ctx->mbd_no_wait = 0;
        if (loop_status != SD_OK) {
            cudaStreamSynchronize(ctx->copy_stream);
            cudaStreamSynchronize(ctx->stream);
            return loop_status;
        }
        return gather_i64_device(ctx, j == 2 ? acc2 : acc3, d_q, nq, d_out);
    };
    return call(ctx, who, X, count_out, true, stage, run);
}

// [rows, colsA] (ldA) next to [rows, colsB] (ldB) -> dense device [rows, colsA + colsB]
static int upload_pooled(sd_ctx *ctx, cudaMemcpyKind kind, const double *A, i64 colsA, i64 ldA, const double *B,
                         i64 colsB, i64 ldB, i64 rows, double **d) {
    const i64 ld = colsA + colsB;
    SD_TRY(ctx->buf[BUF_IN].reserve((size_t)(rows * ld > 0 ? rows * ld : 1) * sizeof(double)));
    *d = ctx->buf[BUF_IN].as<double>();
    if (rows > 0 && colsA > 0)
        SD_CUDA(cudaMemcpy2DAsync(*d, (size_t)ld * sizeof(double), A, (size_t)ldA * sizeof(double),
                                  (size_t)colsA * sizeof(double), (size_t)rows, kind, ctx->stream));
    if (rows > 0 && colsB > 0)
        SD_CUDA(cudaMemcpy2DAsync(*d + colsA, (size_t)ld * sizeof(double), B, (size_t)ldB * sizeof(double),
                                  (size_t)colsB * sizeof(double), (size_t)rows, kind, ctx->stream));
    return SD_OK;
}

// point clouds: [S; Y] rows to BUF_IN, room for the query ids nS .. nS + nY - 1 in BUF_MISC
static int upload_cloud(sd_ctx *ctx, const double *S, i64 nS, int d, const double *Y, i64 nY, double **dP,
                        i64 **d_q) {
    SD_TRY(upload_pooled(ctx, cudaMemcpyHostToDevice, S, nS * d, nS * d, Y, nY * d, nY * d, 1, dP));
    SD_TRY(ctx->buf[BUF_MISC].reserve((size_t)(nY > 0 ? nY : 1) * sizeof(i64)));
    *d_q = ctx->buf[BUF_MISC].as<i64>();
    return SD_OK;
}

// on the device: every point of the pooled cloud finite-checked, then the query ids
static int cloud_queries(sd_ctx *ctx, const double *dP, i64 nS, int d, i64 nY, i64 *d_q) {
    SD_TRY(finite_check_device(ctx, dP, 1, (nS + nY) * d, (nS + nY) * d));
    return iota_from_device(ctx, d_q, nY, nS);
}

// random projection depths (K12, projection.cu).  The directions are small host memory in every variant: checked
// here (finite, non-zero rows), then uploaded to BUF_MISC.
static int upload_directions(sd_ctx *ctx, const double *U, i64 K, int d, const double **dU, const char *who) {
    SD_REQUIRE(U, "%s: NULL directions", who);
    SD_REQUIRE(K >= 1 && d >= 1, "%s: bad sizes K=%lld d=%d", who, (long long)K, d);
    for (i64 k = 0; k < K; ++k) {
        bool nonzero = false;
        for (int c = 0; c < d; ++c) {
            const double u = U[k * d + c];
            SD_REQUIRE(isfinite(u), "%s: direction %lld is not finite", who, (long long)k);
            nonzero |= u != 0.0;
        }
        SD_REQUIRE(nonzero, "%s: direction %lld is zero", who, (long long)k);
    }
    SD_TRY(ctx->buf[BUF_MISC].reserve((size_t)K * d * sizeof(double)));
    double *p = ctx->buf[BUF_MISC].as<double>();
    SD_CUDA(cudaMemcpyAsync(p, U, (size_t)K * d * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    *dU = p;
    return SD_OK;
}

// spatial depth (K14): [S; Y] as dense device rows [nS + nY, F] (Y may be empty).  SD_LAYOUT_TN memory (curves are
// columns, [F, n]) is pooled as [F, nS + nY] and transposed once the kernel phase has begun.
static int upload_curves(Staging &s, const double *S, i64 nS, const double *Y, i64 nY, i64 F, int layout,
                         const double **dP) {
    double *d = nullptr;
    if (layout == SD_LAYOUT_NT) {
        SD_TRY(upload_pooled(s.ctx, cudaMemcpyHostToDevice, S, nS * F, nS * F, Y, nY * F, nY * F, 1, &d));
    } else {
        SD_TRY(upload_pooled(s.ctx, cudaMemcpyHostToDevice, S, nS, nS, Y, nY, nY, F, &d));
        s.nt = d;
        s.nt_rows = F;
        s.nt_cols = nS + nY;
        SD_TRY(s.ctx->buf[BUF_IN2].reserve((size_t)(nS + nY) * F * sizeof(double)));
        d = s.nt_out = s.ctx->buf[BUF_IN2].as<double>();
    }
    *dP = d;
    return SD_OK;
}

}  // namespace sd

using namespace sd;

extern "C" {

// ---------------------------------------------------------------------------------------------
// band depth
// ---------------------------------------------------------------------------------------------
static int band_depth_call(sd_ctx *ctx, const double *X, i64 T, i64 n, i64 ld, int layout, const int64_t *query_idx,
                           i64 nq, int j, int relax, int64_t *count, bool dev, const char *who) {
    SD_TRY(check_matrix(who, T, n, ld, layout));
    SD_REQUIRE(nq >= 0, "%s: bad sizes nq=%lld", who, (long long)nq);
    SD_REQUIRE(query_idx || nq == n, "%s: query_idx == NULL requires nq == n", who);
    // Large relaxed inputs: the H2D copy (PCIe) is ~7x longer than the ranking, and the relaxed numerator is
    // additive over time rows -> stream the matrix in row blocks, copy of block k+1 overlapping ranking of k.
    if (!dev && relax && layout == SD_LAYOUT_TN && (j == 2 || j == 3) && T >= 16 &&
        (size_t)T * n * sizeof(double) >= (64u << 20))
        return band_depth_pipelined(ctx, X, T, n, ld, query_idx, nq, j, count, who);
    const double *dX = X;
    const i64 *d_q = (const i64 *)query_idx;
    i64 *d_count = (i64 *)count;
    return call(ctx, who, X, count, !dev, [&](Staging &s) -> int {
        if (dev) return SD_OK;
        SD_TRY(s.upload_tn(X, T, n, ld, layout, &dX));
        ld = n;
        SD_TRY(upload_queries(ctx, query_idx, nq, n, &d_q, who));
        return s.output(BUF_OUT, count, nq, &d_count);
    }, [&] { return band_depth_device(ctx, dX, T, n, ld, d_q, nq, j, relax, d_count); }, dev && relax);
}

int sd_band_depth_f64(sd_ctx *ctx, const double *X, int64_t T, int64_t n, int64_t ld, int layout,
                      const int64_t *query_idx, int64_t nq, int j, int relax, int64_t *count_out) {
    return band_depth_call(ctx, X, T, n, ld, layout, query_idx, nq, j, relax, count_out, false, "sd_band_depth_f64");
}

int sd_band_depth_f64_dev(sd_ctx *ctx, const double *dX, int64_t T, int64_t n, int64_t ld,
                          const int64_t *d_query_idx, int64_t nq, int j, int relax, int64_t *d_count_out) {
    return band_depth_call(ctx, dX, T, n, ld, SD_LAYOUT_TN, d_query_idx, nq, j, relax, d_count_out, true,
                           "sd_band_depth_f64_dev");
}

int sd_band_ranks_f64(sd_ctx *ctx, const double *X, int64_t T, int64_t n, int64_t ld, int layout,
                      int32_t *below_out, int32_t *above_out) {
    const char *who = "sd_band_ranks_f64";
    SD_REQUIRE(above_out != nullptr, "%s: above_out is NULL", who);
    SD_TRY(check_matrix(who, T, n, ld, layout));
    const double *dX = nullptr;
    int *d_b = nullptr;
    return call(ctx, who, X, below_out, true, [&](Staging &s) -> int {
        SD_TRY(s.upload_tn(X, T, n, ld, layout, &dX));
        SD_TRY(ctx->buf[BUF_OUT].reserve((size_t)T * n * 2 * sizeof(int)));
        d_b = ctx->buf[BUF_OUT].as<int>();
        s.download(below_out, d_b, (size_t)T * n * sizeof(int));
        s.download(above_out, d_b + (size_t)T * n, (size_t)T * n * sizeof(int));
        return SD_OK;
    }, [&] { return rank_rows_device(ctx, dX, T, n, n, d_b, d_b + (size_t)T * n); });
}

int sd_band_depth_batched_f64(sd_ctx *ctx, const double *X, int64_t T, int64_t n, int64_t ld,
                              const uint8_t *membership, int64_t B, const int64_t *queries, int64_t nqb, int j,
                              int relax, int64_t *count_out) {
    const char *who = "sd_band_depth_batched_f64";
    SD_REQUIRE(membership && queries, "%s: NULL membership/queries", who);
    SD_REQUIRE(T >= 1 && n >= 1 && B >= 0 && nqb >= 1 && ld >= n, "%s: bad sizes", who);
    std::vector<i64> cols, offs, qloc;  // member lists and query positions inside each batch
    bool uniform = false;
    i64 m0 = 0;
    double *dX = nullptr;
    i64 *d_cols = nullptr, *d_ql = nullptr, *d_out = nullptr;
    const auto stage = [&](Staging &s) -> int {
        offs.assign((size_t)B + 1, 0);
        qloc.resize((size_t)(B * nqb));
        std::vector<i64> pos((size_t)n);
        for (i64 b = 0; b < B; ++b) {
            const uint8_t *mb = membership + b * n;
            i64 m = 0;
            for (i64 c = 0; c < n; ++c) {
                pos[(size_t)c] = -1;
                if (mb[c]) {
                    pos[(size_t)c] = m++;
                    cols.push_back(c);
                }
            }
            offs[(size_t)b + 1] = offs[(size_t)b] + m;
            for (i64 i = 0; i < nqb; ++i) {
                const i64 g = queries[b * nqb + i];
                SD_REQUIRE(g >= 0 && g < n && pos[(size_t)g] >= 0, "%s: query %lld of batch %lld is not a member",
                           who, (long long)g, (long long)b);
                qloc[(size_t)(b * nqb + i)] = pos[(size_t)g];
            }
        }
        // relaxed depth with equally sized batches (permutation tests): ALL batches go through the rank pipeline as
        // one matrix of B*T rows whose row groups accumulate separately -- a handful of launches instead of ~10 per
        // batch
        const bool strict_match = !relax && j == 2 && (ctx->bd_impl == SD_BD_AUTO || ctx->bd_impl == SD_BD_MATCH);
        uniform = B > 1 && ((relax != 0 && (j == 2 || j == 3)) || strict_match);
        m0 = B > 0 ? offs[1] - offs[0] : 0;
        for (i64 b = 0; b < B && uniform; ++b) uniform = offs[(size_t)b + 1] - offs[(size_t)b] == m0;
        if (uniform && !relax && !bd_match_supported(T, m0)) uniform = false;
        if (uniform && m0 >= 1 && relax && relaxed_overflows(T, m0 - 1, j))
            uniform = false;  // let the per-batch path report the overflow
        if (uniform && m0 >= 1 && relax)
            for (i64 b = 0; b < B; ++b)  // flat index of every query in the [B][m0] accumulator
                for (i64 i = 0; i < nqb; ++i) qloc[(size_t)(b * nqb + i)] += b * m0;
        SD_TRY(upload_matrix(ctx, BUF_IN, X, T, n, ld, &dX));
        SD_TRY(ctx->buf[BUF_AUX].reserve((cols.size() + 1) * sizeof(i64)));
        SD_TRY(ctx->buf[BUF_MISC].reserve((qloc.size() + 1) * sizeof(i64)));
        SD_TRY(ctx->buf[BUF_OUT].reserve((qloc.size() + 1) * sizeof(i64)));
        d_cols = ctx->buf[BUF_AUX].as<i64>();
        d_ql = ctx->buf[BUF_MISC].as<i64>();
        d_out = ctx->buf[BUF_OUT].as<i64>();
        // cols / qloc are pageable host vectors: these async copies are staged synchronously
        if (!cols.empty())
            SD_CUDA(cudaMemcpyAsync(d_cols, cols.data(), cols.size() * sizeof(i64), cudaMemcpyHostToDevice,
                                    ctx->stream));
        if (!qloc.empty())
            SD_CUDA(cudaMemcpyAsync(d_ql, qloc.data(), qloc.size() * sizeof(i64), cudaMemcpyHostToDevice,
                                    ctx->stream));
        s.download(count_out, d_out, qloc.size() * sizeof(i64));
        return SD_OK;
    };
    const auto run = [&]() -> int {
        if (uniform && m0 >= 1) {
            // batches per pass: the gathered matrix stays below ~1 GB
            i64 BB = (i64)((1ull << 30) / ((size_t)T * m0 * sizeof(double)));
            if (BB < 1) BB = 1;
            if (BB > B) BB = B;
            SD_TRY(ctx->buf[BUF_IN2].reserve((size_t)BB * T * m0 * sizeof(double)));
            SD_TRY(ctx->buf[BUF_ACC].reserve((size_t)B * m0 * 2 * sizeof(i64)));
            double *dXg = ctx->buf[BUF_IN2].as<double>();
            i64 *acc2 = ctx->buf[BUF_ACC].as<i64>(), *acc3 = acc2 + B * m0;
            for (i64 b0 = 0; b0 < B; b0 += BB) {
                const i64 nb = B - b0 < BB ? B - b0 : BB;
                SD_TRY(compact_batches_device(ctx, dX, T, n, d_cols + b0 * m0, m0, nb, dXg));
                if (relax) {
                    SD_TRY(mbd_all_device(ctx, dXg, nb * T, m0, m0, acc2 + b0 * m0, j == 3 ? acc3 + b0 * m0 : nullptr,
                                          false, T));
                } else {  // strict: sign-vector matcher over all sub-populations of the pass
                    ctx->last.bd_impl_used = SD_BD_MATCH;
                    SD_TRY(bd_strict_match_batched_device(ctx, dXg, nb, T, m0, d_ql + b0 * nqb, nqb, d_out + b0 * nqb,
                                                          strict_enumerate));
                }
            }
            if (relax) SD_TRY(gather_i64_device(ctx, j == 2 ? acc2 : acc3, d_ql, (i64)qloc.size(), d_out));
            return SD_OK;
        }
        SD_TRY(ctx->buf[BUF_IN2].reserve((size_t)T * n * sizeof(double)));
        double *dXb = ctx->buf[BUF_IN2].as<double>();
        for (i64 b = 0; b < B; ++b) {
            const i64 m = offs[(size_t)b + 1] - offs[(size_t)b];
            SD_TRY(compact_columns_device(ctx, dX, T, n, d_cols + offs[(size_t)b], m, dXb));
            SD_TRY(band_depth_device(ctx, dXb, T, m, m, d_ql + b * nqb, nqb, j, relax, d_out + b * nqb));
        }
        return SD_OK;
    };
    return call(ctx, who, X, count_out, true, stage, run);
}

// ---------------------------------------------------------------------------------------------
// out-of-sample depth: sample and new observations are pooled on the device (sample first), see oos.cu
// ---------------------------------------------------------------------------------------------
static int band_depth_oos_call(sd_ctx *ctx, const double *S, i64 T, i64 nS, i64 ldS, const double *Y, i64 nY,
                               i64 ldY, int j, int relax, int64_t *count, bool dev, const char *who) {
    SD_REQUIRE(Y || nY == 0, "%s: NULL Y", who);
    SD_REQUIRE(T >= 1 && nS >= 1 && nY >= 0 && ldS >= nS && ldY >= nY, "%s: bad sizes", who);
    const double *dX = S;
    i64 ld = ldS;
    i64 *d_count = (i64 *)count;
    double *pooled = nullptr;
    return call(ctx, who, S, count, !dev, [&](Staging &s) -> int {
        if (dev) return SD_OK;
        SD_TRY(upload_pooled(ctx, cudaMemcpyHostToDevice, S, nS, ldS, Y, nY, ldY, T, &pooled));
        dX = pooled;
        ld = nS + nY;
        return s.output(BUF_OUT, count, nY, &d_count);
    }, [&]() -> int {
        if (dev && nY > 0 && !(Y == S + nS && ldY == ldS)) {  // not already the columns after the sample: pool them
            SD_TRY(upload_pooled(ctx, cudaMemcpyDeviceToDevice, S, nS, ldS, Y, nY, ldY, T, &pooled));
            dX = pooled;
            ld = nS + nY;
        }
        return band_depth_oos_device(ctx, dX, T, nS, nY, ld, j, relax, d_count);
    });
}

int sd_band_depth_oos_f64(sd_ctx *ctx, const double *S, int64_t T, int64_t nS, int64_t ldS, const double *Y,
                          int64_t nY, int64_t ldY, int j, int relax, int64_t *count_out) {
    return band_depth_oos_call(ctx, S, T, nS, ldS, Y, nY, ldY, j, relax, count_out, false, "sd_band_depth_oos_f64");
}

int sd_band_depth_oos_f64_dev(sd_ctx *ctx, const double *dS, int64_t T, int64_t nS, int64_t ldS, const double *dY,
                              int64_t nY, int64_t ldY, int j, int relax, int64_t *d_count_out) {
    return band_depth_oos_call(ctx, dS, T, nS, ldS, dY, nY, ldY, j, relax, d_count_out, true,
                               "sd_band_depth_oos_f64_dev");
}

// a fitted reference: sorted sample rows, and out-of-sample counts from them (reference.cu)
int sd_band_sort_rows_f64_dev(sd_ctx *ctx, const double *dX, int64_t T, int64_t nS, int64_t ld,
                              double *d_sorted_out) {
    const char *who = "sd_band_sort_rows_f64_dev";
    SD_REQUIRE(T >= 1 && nS >= 1 && ld >= nS, "%s: bad sizes", who);
    return call(ctx, who, dX, d_sorted_out, false, no_stage,
                [&] { return sort_rows_device(ctx, dX, T, nS, ld, d_sorted_out); });
}

int sd_band_depth_sorted_f64_dev(sd_ctx *ctx, const double *d_sorted, int64_t T, int64_t nS, const double *dY,
                                 int64_t nY, int64_t ldY, int J, int64_t *d_count_out) {
    const char *who = "sd_band_depth_sorted_f64_dev";
    SD_REQUIRE(dY || nY == 0, "%s: NULL Y", who);
    SD_REQUIRE(T >= 1 && nS >= 1 && nY >= 0 && ldY >= nY, "%s: bad sizes", who);
    return call(ctx, who, d_sorted, d_count_out, false, no_stage,
                [&] { return depth_sorted_device(ctx, d_sorted, T, nS, dY, nY, ldY, J, (i64 *)d_count_out); });
}

int sd_pointcloud_simplicial_oos_f64(sd_ctx *ctx, const double *S, int64_t nS, int d, const double *Y, int64_t nY,
                                     double tol, int64_t *count_out) {
    const char *who = "sd_pointcloud_simplicial_oos_f64";
    SD_REQUIRE(Y || nY == 0, "%s: NULL Y", who);
    SD_REQUIRE(nS >= 1 && nY >= 0, "%s: bad sizes", who);
    SD_REQUIRE(d >= 1 && d <= 3, "%s: d=%d not supported (1..3)", who, d);
    SD_REQUIRE(tol >= 0.0, "%s: tol must be >= 0", who);
    double *dP = nullptr;
    i64 *d_q = nullptr, *d_out = nullptr;
    return call(ctx, who, S, count_out, true, [&](Staging &s) -> int {
        SD_TRY(s.output(BUF_OUT, count_out, nY, &d_out));
        return upload_cloud(ctx, S, nS, d, Y, nY, &dP, &d_q);
    }, [&]() -> int {
        SD_TRY(cloud_queries(ctx, dP, nS, d, nY, d_q));
        return simplicial_device(ctx, dP, nS + 1, d, d_q, nY, tol, d_out, true);
    });
}

int sd_pointcloud_l1_oos_f64(sd_ctx *ctx, const double *S, int64_t nS, int d, const double *Y, int64_t nY,
                             double *depth_out) {
    const char *who = "sd_pointcloud_l1_oos_f64";
    SD_REQUIRE(Y || nY == 0, "%s: NULL Y", who);
    SD_REQUIRE(nS >= 1 && nY >= 0, "%s: bad sizes", who);
    SD_REQUIRE(d >= 1 && d <= 16, "%s: d=%d not supported (1..16)", who, d);
    double *dP = nullptr, *d_out = nullptr;
    i64 *d_q = nullptr;
    return call(ctx, who, S, depth_out, true, [&](Staging &s) -> int {
        SD_TRY(s.output(BUF_OUT, depth_out, nY, &d_out));
        return upload_cloud(ctx, S, nS, d, Y, nY, &dP, &d_q);
    }, [&]() -> int {
        SD_TRY(cloud_queries(ctx, dP, nS, d, nY, d_q));
        return l1_device(ctx, dP, nS, d, d_q, nY, d_out, nS + 1);
    });
}

// ---------------------------------------------------------------------------------------------
// outlier detection: per-curve rank sums and masked envelopes, see outliers.cu
// ---------------------------------------------------------------------------------------------
static int rank_sums_call(sd_ctx *ctx, const double *X, i64 T, i64 n, i64 ld, int layout, int64_t *q, int64_t *below,
                          int64_t *above, bool dev, const char *who) {
    SD_REQUIRE(below, "%s: NULL below_sum_out", who);
    SD_TRY(check_matrix(who, T, n, ld, layout));
    const double *dX = X;
    i64 *d_q = (i64 *)q, *d_b = (i64 *)below, *d_a = (i64 *)above;
    return call(ctx, who, X, q, !dev, [&](Staging &s) -> int {
        if (dev) return SD_OK;
        SD_TRY(s.upload_tn(X, T, n, ld, layout, &dX));
        ld = n;
        SD_TRY(ctx->buf[BUF_OUT].reserve((size_t)n * 3 * sizeof(i64)));
        d_q = ctx->buf[BUF_OUT].as<i64>();
        d_b = d_q + n;
        d_a = above ? d_b + n : nullptr;
        s.download(q, d_q, (size_t)n * sizeof(i64));
        s.download(below, d_b, (size_t)n * sizeof(i64));
        s.download(above, d_a, (size_t)n * sizeof(i64));
        return SD_OK;
    }, [&] { return rank_sums_device(ctx, dX, T, n, ld, d_q, d_b, d_a); });
}

int sd_band_rank_sums_f64(sd_ctx *ctx, const double *X, int64_t T, int64_t n, int64_t ld, int layout, int64_t *q_out,
                          int64_t *below_sum_out, int64_t *above_sum_out) {
    return rank_sums_call(ctx, X, T, n, ld, layout, q_out, below_sum_out, above_sum_out, false,
                          "sd_band_rank_sums_f64");
}

int sd_band_rank_sums_f64_dev(sd_ctx *ctx, const double *dX, int64_t T, int64_t n, int64_t ld, int64_t *d_q_out,
                              int64_t *d_below_sum_out, int64_t *d_above_sum_out) {
    return rank_sums_call(ctx, dX, T, n, ld, SD_LAYOUT_TN, d_q_out, d_below_sum_out, d_above_sum_out, true,
                          "sd_band_rank_sums_f64_dev");
}

static int envelope_call(sd_ctx *ctx, const double *X, i64 T, i64 n, i64 ld, int layout, const uint8_t *member,
                         double factor, double *lower, double *upper, int64_t *outside, bool dev, const char *who) {
    SD_REQUIRE(member && upper, "%s: NULL member or upper_out", who);
    SD_TRY(check_matrix(who, T, n, ld, layout));
    const double *dX = X;
    const uint8_t *d_member = member;
    double *d_lo = lower, *d_hi = upper;
    i64 *d_out = (i64 *)outside;
    return call(ctx, who, X, lower, !dev, [&](Staging &s) -> int {
        if (dev) return SD_OK;
        SD_TRY(s.upload_tn(X, T, n, ld, layout, &dX));
        ld = n;
        // lower | upper | outside | member
        SD_TRY(ctx->buf[BUF_OUT].reserve((size_t)(2 * T + n) * 8 + (size_t)n));
        d_lo = ctx->buf[BUF_OUT].as<double>();
        d_hi = d_lo + T;
        d_out = outside ? reinterpret_cast<i64 *>(d_hi + T) : nullptr;
        uint8_t *dm = reinterpret_cast<uint8_t *>(d_hi + T + n);
        SD_CUDA(cudaMemcpyAsync(dm, member, (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
        d_member = dm;
        s.download(lower, d_lo, (size_t)T * 8);
        s.download(upper, d_hi, (size_t)T * 8);
        s.download(outside, d_out, (size_t)n * 8);
        return SD_OK;
    }, [&] { return envelope_device(ctx, dX, T, n, ld, d_member, factor, d_lo, d_hi, d_out); });
}

int sd_band_envelope_f64(sd_ctx *ctx, const double *X, int64_t T, int64_t n, int64_t ld, int layout,
                         const uint8_t *member, double factor, double *lower_out, double *upper_out,
                         int64_t *outside_out) {
    return envelope_call(ctx, X, T, n, ld, layout, member, factor, lower_out, upper_out, outside_out, false,
                         "sd_band_envelope_f64");
}

int sd_band_envelope_f64_dev(sd_ctx *ctx, const double *dX, int64_t T, int64_t n, int64_t ld,
                             const uint8_t *d_member, double factor, double *d_lower_out, double *d_upper_out,
                             int64_t *d_outside_out) {
    return envelope_call(ctx, dX, T, n, ld, SD_LAYOUT_TN, d_member, factor, d_lower_out, d_upper_out, d_outside_out,
                         true, "sd_band_envelope_f64_dev");
}

// extremal depth: pointwise extremities of a block of rows, numerators from the full matrix (extremal.cu)
int sd_band_extremity_f64_dev(sd_ctx *ctx, const double *dX, int64_t T, int64_t n, int64_t ld, int32_t *d_m_out) {
    const char *who = "sd_band_extremity_f64_dev";
    SD_TRY(check_matrix(who, T, n, ld, SD_LAYOUT_TN));
    return call(ctx, who, dX, d_m_out, false, no_stage,
                [&] { return extremity_device(ctx, dX, T, n, ld, (int *)d_m_out); });
}

int sd_extremal_depth_dev(sd_ctx *ctx, const int32_t *d_m, int64_t T, int64_t n, int64_t *d_num_out) {
    const char *who = "sd_extremal_depth_dev";
    SD_REQUIRE(T >= 1 && n >= 1, "%s: bad sizes T=%lld n=%lld", who, (long long)T, (long long)n);
    return call(ctx, who, d_m, d_num_out, false, no_stage,
                [&] { return extremal_depth_device(ctx, (const int *)d_m, T, n, (i64 *)d_num_out); });
}

// ---------------------------------------------------------------------------------------------
// multivariate curves and point clouds
// ---------------------------------------------------------------------------------------------
int sd_simplex_depth_f64(sd_ctx *ctx, const double *F, int64_t N, int64_t T, int d, const int64_t *query_idx,
                         int64_t nq, int relax, double tol, int64_t *count_out) {
    const char *who = "sd_simplex_depth_f64";
    SD_REQUIRE(N >= 1 && T >= 1 && nq >= 0, "%s: bad sizes", who);
    SD_REQUIRE(d >= 1 && d <= 3, "%s: d=%d not supported (1..3)", who, d);
    SD_REQUIRE(tol >= 0.0, "%s: tol must be >= 0", who);
    double *dF = nullptr;
    const i64 *d_q = nullptr;
    i64 *d_out = nullptr;
    return call(ctx, who, F, count_out, true, [&](Staging &s) -> int {
        SD_TRY(upload_matrix(ctx, BUF_IN, F, 1, N * T * d, N * T * d, &dF));
        SD_TRY(upload_queries(ctx, query_idx, nq, N, &d_q, who));
        return s.output(BUF_OUT, count_out, nq, &d_out);
    }, [&] { return simplex_depth_device(ctx, dF, N, T, d, d_q, nq, relax, tol, d_out); });
}

int sd_pointcloud_simplicial_f64(sd_ctx *ctx, const double *P, int64_t n, int d, const int64_t *query_idx,
                                 int64_t nq, double tol, int64_t *count_out) {
    const char *who = "sd_pointcloud_simplicial_f64";
    SD_REQUIRE(n >= 1 && nq >= 0, "%s: bad sizes", who);
    SD_REQUIRE(d >= 1 && d <= 3, "%s: d=%d not supported (1..3)", who, d);
    SD_REQUIRE(tol >= 0.0, "%s: tol must be >= 0", who);
    double *dP = nullptr;
    const i64 *d_q = nullptr;
    i64 *d_out = nullptr;
    return call(ctx, who, P, count_out, true, [&](Staging &s) -> int {
        SD_TRY(upload_matrix(ctx, BUF_IN, P, 1, n * d, n * d, &dP));
        SD_TRY(upload_queries(ctx, query_idx, nq, n, &d_q, who));
        return s.output(BUF_OUT, count_out, nq, &d_out);
    }, [&] { return simplicial_device(ctx, dP, n, d, d_q, nq, tol, d_out); });
}

int sd_pointcloud_l1_f64(sd_ctx *ctx, const double *P, int64_t n, int d, const int64_t *query_idx, int64_t nq,
                         double *depth_out) {
    const char *who = "sd_pointcloud_l1_f64";
    SD_REQUIRE(n >= 1 && nq >= 0, "%s: bad sizes", who);
    SD_REQUIRE(d >= 1 && d <= 16, "%s: d=%d not supported (1..16)", who, d);
    double *dP = nullptr, *d_out = nullptr;
    const i64 *d_q = nullptr;
    return call(ctx, who, P, depth_out, true, [&](Staging &s) -> int {
        SD_TRY(upload_matrix(ctx, BUF_IN, P, 1, n * d, n * d, &dP));
        SD_TRY(upload_queries(ctx, query_idx, nq, n, &d_q, who));
        return s.output(BUF_OUT, depth_out, nq, &d_out);
    }, [&] { return l1_device(ctx, dP, n, d, d_q, nq, d_out); });
}

int sd_pointcloud_oja_f64(sd_ctx *ctx, const double *P, int64_t n, int d, const int64_t *query_idx, int64_t nq,
                          const int64_t *pool, int64_t npool, double hull_volume, double *out) {
    const char *who = "sd_pointcloud_oja_f64";
    SD_REQUIRE(n >= 1 && nq >= 0 && npool >= 0, "%s: bad sizes", who);
    SD_REQUIRE(d == 2 || d == 3, "%s: d=%d not supported (2 or 3)", who, d);
    SD_REQUIRE(pool || npool == n, "%s: pool == NULL requires npool == n", who);
    double *dP = nullptr, *d_out = nullptr;
    const i64 *d_q = nullptr, *d_pool = nullptr;
    return call(ctx, who, P, out, true, [&](Staging &s) -> int {
        SD_TRY(upload_matrix(ctx, BUF_IN, P, 1, n * d, n * d, &dP));
        SD_TRY(upload_queries(ctx, query_idx, nq, n, &d_q, who));
        if (pool) {
            for (i64 i = 0; i < npool; ++i)
                SD_REQUIRE(pool[i] >= 0 && pool[i] < n, "%s: pool[%lld] out of range", who, (long long)i);
            SD_TRY(ctx->buf[BUF_AUX].reserve((size_t)(npool > 0 ? npool : 1) * sizeof(i64)));
            if (npool > 0)
                SD_CUDA(cudaMemcpyAsync(ctx->buf[BUF_AUX].p, pool, (size_t)npool * sizeof(i64),
                                        cudaMemcpyHostToDevice, ctx->stream));
            d_pool = ctx->buf[BUF_AUX].as<i64>();
        }
        return s.output(BUF_OUT, out, nq, &d_out);
    }, [&] { return oja_device(ctx, dP, n, d, d_q, nq, d_pool, npool, hull_volume, d_out); });
}

int sd_pointcloud_blocks_f64(sd_ctx *ctx, const double *P, int64_t n, int d, const int64_t *member,
                             const int64_t *block_off, const int64_t *query_pos, int64_t B, int kind, double tol,
                             const double *hull_volume, double *out) {
    const char *who = "sd_pointcloud_blocks_f64";
    SD_REQUIRE(n >= 1 && B >= 0 && member && block_off && query_pos, "%s: bad arguments", who);
    SD_REQUIRE(d >= 1 && d <= 3, "%s: d=%d not supported (1..3)", who, d);
    SD_REQUIRE(kind >= 0 && kind <= 2, "%s: kind=%d (0 simplicial, 1 l1, 2 oja)", who, kind);
    SD_REQUIRE(kind != 2 || (hull_volume && d >= 2), "%s: oja needs d in (2, 3) and hull volumes", who);
    SD_REQUIRE(tol >= 0.0, "%s: tol must be >= 0", who);
    SD_REQUIRE(block_off[0] == 0, "%s: block_off[0] must be 0", who);
    for (i64 b = 0; b < B; ++b) {
        const i64 m = block_off[b + 1] - block_off[b];
        SD_REQUIRE(m >= 1 && m * d <= 4096, "%s: block %lld has %lld members (1 .. %d supported)", who, (long long)b,
                   (long long)m, 4096 / d);
        SD_REQUIRE(query_pos[b] >= 0 && query_pos[b] < m, "%s: query_pos[%lld] out of range", who, (long long)b);
    }
    const i64 total = B > 0 ? block_off[B] : 0;
    for (i64 i = 0; i < total; ++i)
        SD_REQUIRE(member[i] >= 0 && member[i] < n, "%s: member[%lld] out of range", who, (long long)i);
    double *dP = nullptr, *d_vol = nullptr, *d_out = nullptr;
    i64 *d_member = nullptr, *d_off = nullptr, *d_qpos = nullptr;
    return call(ctx, who, P, out, true, [&](Staging &s) -> int {
        SD_TRY(upload_matrix(ctx, BUF_IN, P, 1, n * d, n * d, &dP));
        // member | block_off | query_pos | hull volumes | out, in one workspace buffer
        const size_t words = (size_t)total + (size_t)(B + 1) + (size_t)B + (size_t)B + (size_t)B + 8;
        SD_TRY(ctx->buf[BUF_AUX].reserve(words * 8));
        d_member = ctx->buf[BUF_AUX].as<i64>();
        d_off = d_member + total;
        d_qpos = d_off + (B + 1);
        d_vol = reinterpret_cast<double *>(d_qpos + B);
        d_out = d_vol + B;
        if (total > 0)
            SD_CUDA(cudaMemcpyAsync(d_member, member, (size_t)total * 8, cudaMemcpyHostToDevice, ctx->stream));
        SD_CUDA(cudaMemcpyAsync(d_off, block_off, (size_t)(B + 1) * 8, cudaMemcpyHostToDevice, ctx->stream));
        if (B > 0) {
            SD_CUDA(cudaMemcpyAsync(d_qpos, query_pos, (size_t)B * 8, cudaMemcpyHostToDevice, ctx->stream));
            if (hull_volume)
                SD_CUDA(cudaMemcpyAsync(d_vol, hull_volume, (size_t)B * 8, cudaMemcpyHostToDevice, ctx->stream));
        }
        s.download(out, d_out, (size_t)B * 8);
        return SD_OK;
    }, [&] {
        return cloud_blocks_device(ctx, dP, d, d_member, d_off, d_qpos, B, kind, tol, hull_volume ? d_vol : nullptr,
                                   d_out);
    });
}

// halfspace (Tukey) depth numerators (K11): d = 1 from K1's ranks (halfspace.cu), d = 2 from the angular keys
// (hs_reduce_kernel, simplicial_count.cu).  Every value is finite-checked whatever the queries; the row lengths are
// checked by the rank pipeline (n < 2^31) and the angular counting (2n < 2^31).

int sd_pointcloud_halfspace_f64(sd_ctx *ctx, const double *P, int64_t n, int d, const int64_t *query_idx,
                                int64_t nq, int64_t *count_out) {
    const char *who = "sd_pointcloud_halfspace_f64";
    SD_REQUIRE(n >= 1 && nq >= 0, "%s: bad sizes", who);
    if (d != 1 && d != 2) {
        set_error("%s: d=%d not supported (1 or 2)", who, d);
        return SD_ERR_UNSUPPORTED;
    }
    double *dP = nullptr;
    const i64 *d_q = nullptr;
    i64 *d_out = nullptr;
    return call(ctx, who, P, count_out, true, [&](Staging &s) -> int {
        SD_TRY(upload_matrix(ctx, BUF_IN, P, 1, n * d, n * d, &dP));
        SD_TRY(upload_queries(ctx, query_idx, nq, n, &d_q, who));
        SD_TRY(ctx->buf[BUF_OUT].reserve((size_t)(nq + (d == 1 ? n : 0) + 1) * sizeof(i64)));
        d_out = ctx->buf[BUF_OUT].as<i64>();
        s.download(count_out, d_out, (size_t)nq * sizeof(i64));
        return SD_OK;
    }, [&]() -> int {
        SD_TRY(finite_check_device(ctx, dP, 1, n * d, n * d));
        if (d == 2) return simplicial2_count_device(ctx, dP, n, 2, 1, d_q, nq, 0.0, d_out, -1, SC_HALFSPACE);
        // one row of n values: every point's numerator, then the queries'
        i64 *d_all = d_out + nq;
        SD_TRY(halfspace1_device(ctx, dP, 1, n, n, d_all));
        return gather_i64_device(ctx, d_all, d_q, nq, d_out);
    });
}

int sd_functional_halfspace_f64(sd_ctx *ctx, const double *F, int64_t N, int64_t T, int d, const int64_t *query_idx,
                                int64_t nq, int64_t *count_out) {
    const char *who = "sd_functional_halfspace_f64";
    SD_REQUIRE(N >= 1 && T >= 1 && nq >= 0, "%s: bad sizes", who);
    if (d != 2) {
        set_error("%s: d=%d not supported (2)", who, d);
        return SD_ERR_UNSUPPORTED;
    }
    double *dF = nullptr;
    const i64 *d_q = nullptr;
    i64 *d_out = nullptr;
    return call(ctx, who, F, count_out, true, [&](Staging &s) -> int {
        SD_TRY(upload_matrix(ctx, BUF_IN, F, 1, N * T * d, N * T * d, &dF));
        SD_TRY(upload_queries(ctx, query_idx, nq, N, &d_q, who));
        return s.output(BUF_OUT, count_out, nq, &d_out);
    }, [&]() -> int {
        SD_TRY(finite_check_device(ctx, dF, 1, N * T * d, N * T * d));
        return simplicial2_count_device(ctx, dF, N, 2 * T, T, d_q, nq, 0.0, d_out, -1, SC_HALFSPACE);
    });
}

static int band_halfspace_call(sd_ctx *ctx, const double *X, i64 T, i64 n, i64 ld, int layout, int64_t *count,
                               bool dev, const char *who) {
    SD_TRY(check_matrix(who, T, n, ld, layout));
    const double *dX = X;
    i64 *d_count = (i64 *)count;
    return call(ctx, who, X, count, !dev, [&](Staging &s) -> int {
        if (dev) return SD_OK;
        SD_TRY(s.upload_tn(X, T, n, ld, layout, &dX));
        ld = n;
        return s.output(BUF_OUT, count, n, &d_count);
    }, [&] { return halfspace1_device(ctx, dX, T, n, ld, d_count); });
}

int sd_band_halfspace_f64(sd_ctx *ctx, const double *X, int64_t T, int64_t n, int64_t ld, int layout,
                          int64_t *count_out) {
    return band_halfspace_call(ctx, X, T, n, ld, layout, count_out, false, "sd_band_halfspace_f64");
}

int sd_band_halfspace_f64_dev(sd_ctx *ctx, const double *dX, int64_t T, int64_t n, int64_t ld,
                              int64_t *d_count_out) {
    return band_halfspace_call(ctx, dX, T, n, ld, SD_LAYOUT_TN, d_count_out, true, "sd_band_halfspace_f64_dev");
}

// ---------------------------------------------------------------------------------------------
// random projection depths (K12, projection.cu)
// ---------------------------------------------------------------------------------------------
static int projection_call(sd_ctx *ctx, const double *F, int64_t N, int64_t T, int d, const double *U, int64_t K,
                           ProjKind kind, void *out, double *med_out, double *mad_out, bool dev, const char *who) {
    SD_REQUIRE(N >= 1 && T >= 1 && d >= 1 && K >= 1, "%s: bad sizes N=%lld T=%lld d=%d K=%lld", who, (long long)N,
               (long long)T, d, (long long)K);
    if (N >= (1ll << 31)) {  // the rank pipeline's limit, refused before anything is uploaded
        set_error("%s: N=%lld exceeds 2^31-1", who, (long long)N);
        return SD_ERR_UNSUPPORTED;
    }
    const double *dU = nullptr, *dF = F;
    void *d_out = out;
    return call(ctx, who, F, out, !dev, [&](Staging &s) -> int {
        SD_TRY(upload_directions(ctx, U, K, d, &dU, who));
        if (dev) return SD_OK;
        double *up = nullptr;
        SD_TRY(upload_matrix(ctx, BUF_IN, F, 1, N * T * d, N * T * d, &up));
        dF = up;
        const size_t out_bytes = (size_t)N * (kind == PJ_TUKEY ? 1 : T) * 8;
        SD_TRY(ctx->buf[BUF_OUT].reserve(out_bytes));
        d_out = ctx->buf[BUF_OUT].p;
        s.download(out, d_out, out_bytes);
        return SD_OK;
    }, [&] {
        return projection_device(ctx, dF, N, T, d, N * T * d, dU, K, kind, (i64 *)d_out, (double *)d_out, med_out,
                                 mad_out, dev ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost);
    });
}

int sd_projection_tukey_f64(sd_ctx *ctx, const double *F, int64_t N, int64_t T, int d, const double *U, int64_t K,
                            int64_t *count_out) {
    return projection_call(ctx, F, N, T, d, U, K, PJ_TUKEY, count_out, nullptr, nullptr, false,
                           "sd_projection_tukey_f64");
}

int sd_projection_tukey_f64_dev(sd_ctx *ctx, const double *dF, int64_t N, int64_t T, int d, const double *U,
                                int64_t K, int64_t *d_count_out) {
    return projection_call(ctx, dF, N, T, d, U, K, PJ_TUKEY, d_count_out, nullptr, nullptr, true,
                           "sd_projection_tukey_f64_dev");
}

int sd_projection_outlyingness_f64(sd_ctx *ctx, const double *F, int64_t N, int64_t T, int d, const double *U,
                                   int64_t K, double *o_out, double *med_out, double *mad_out) {
    return projection_call(ctx, F, N, T, d, U, K, PJ_OUTLYING, o_out, med_out, mad_out, false,
                           "sd_projection_outlyingness_f64");
}

int sd_projection_outlyingness_f64_dev(sd_ctx *ctx, const double *dF, int64_t N, int64_t T, int d,
                                       const double *U, int64_t K, double *d_o_out, double *d_med_out,
                                       double *d_mad_out) {
    return projection_call(ctx, dF, N, T, d, U, K, PJ_OUTLYING, d_o_out, d_med_out, d_mad_out, true,
                           "sd_projection_outlyingness_f64_dev");
}

static int band_outlyingness_call(sd_ctx *ctx, const double *X, i64 T, i64 n, i64 ld, int layout, double *o,
                                  double *med, double *mad, bool dev, const char *who) {
    SD_TRY(check_matrix(who, T, n, ld, layout));
    if (n >= (1ll << 31)) {
        set_error("%s: n=%lld exceeds 2^31-1", who, (long long)n);
        return SD_ERR_UNSUPPORTED;
    }
    const double *dX = X;
    double *d_o = o;
    return call(ctx, who, X, o, !dev, [&](Staging &s) -> int {
        if (dev) return SD_OK;
        SD_TRY(s.upload_tn(X, T, n, ld, layout, &dX));
        ld = n;
        return s.output(BUF_OUT, o, T * n, &d_o);
    }, [&] {
        return projection_device(ctx, dX, n, T, 1, ld, nullptr, 1, PJ_OUTLYING, nullptr, d_o, med, mad,
                                 dev ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost);
    });
}

int sd_band_outlyingness_f64(sd_ctx *ctx, const double *X, int64_t T, int64_t n, int64_t ld, int layout,
                             double *o_out, double *med_out, double *mad_out) {
    return band_outlyingness_call(ctx, X, T, n, ld, layout, o_out, med_out, mad_out, false,
                                  "sd_band_outlyingness_f64");
}

int sd_band_outlyingness_f64_dev(sd_ctx *ctx, const double *dX, int64_t T, int64_t n, int64_t ld, double *d_o_out,
                                 double *d_med_out, double *d_mad_out) {
    return band_outlyingness_call(ctx, dX, T, n, ld, SD_LAYOUT_TN, d_o_out, d_med_out, d_mad_out, true,
                                  "sd_band_outlyingness_f64_dev");
}

// ---------------------------------------------------------------------------------------------
// fitted references for random projection depths (K13, reference_proj.cu)
// ---------------------------------------------------------------------------------------------
int sd_projection_sort_rows_f64_dev(sd_ctx *ctx, const double *dF, int64_t nS, int64_t T, int d, const double *U,
                                    int64_t K, double *d_sorted_out) {
    const char *who = "sd_projection_sort_rows_f64_dev";
    SD_REQUIRE(nS >= 1 && T >= 1 && d >= 1 && K >= 1, "%s: bad sizes nS=%lld T=%lld d=%d K=%lld", who,
               (long long)nS, (long long)T, d, (long long)K);
    if (nS >= (1ll << 31)) {  // the rank pipeline's limit, refused before anything is uploaded
        set_error("%s: nS=%lld exceeds 2^31-1", who, (long long)nS);
        return SD_ERR_UNSUPPORTED;
    }
    const double *dU = nullptr;
    return call(ctx, who, dF, d_sorted_out, false,
                [&](Staging &) { return upload_directions(ctx, U, K, d, &dU, who); },
                [&] { return projection_sort_rows_device(ctx, dF, nS, T, d, dU, K, d_sorted_out); });
}

// new observations against a sorted index: U == NULL takes the univariate rows dY [T, nY] (ldY) against K9's index
static int sorted_query_call(sd_ctx *ctx, const double *d_sorted, i64 nS, i64 T, const double *dY, i64 nY, i64 ldY,
                             int d, const double *U, i64 K, ProjKind kind, void *out, const char *who) {
    SD_REQUIRE(dY || nY == 0, "%s: NULL new data", who);
    SD_REQUIRE(nS >= 1 && T >= 1 && nY >= 0 && d >= 1 && K >= 1 && ldY >= nY,
               "%s: bad sizes nS=%lld T=%lld nY=%lld d=%d K=%lld ldY=%lld", who, (long long)nS, (long long)T,
               (long long)nY, d, (long long)K, (long long)ldY);
    if (nS + 1 >= (1ll << 31)) {
        set_error("%s: nS + 1 = %lld exceeds 2^31-1", who, (long long)(nS + 1));
        return SD_ERR_UNSUPPORTED;
    }
    const double *dU = nullptr;
    return call(ctx, who, d_sorted, out, false,
                [&](Staging &) { return U ? upload_directions(ctx, U, K, d, &dU, who) : SD_OK; },
                [&] {
                    return projection_sorted_device(ctx, d_sorted, nS, T, dY, nY, ldY, d, dU, K, kind, (i64 *)out,
                                                    (double *)out);
                });
}

int sd_projection_tukey_sorted_f64_dev(sd_ctx *ctx, const double *d_sorted, int64_t nS, int64_t T,
                                       const double *dF_new, int64_t nY, int d, const double *U, int64_t K,
                                       int64_t *d_count_out) {
    return sorted_query_call(ctx, d_sorted, nS, T, dF_new, nY, nY, d, U, K, PJ_TUKEY, d_count_out,
                             "sd_projection_tukey_sorted_f64_dev");
}

int sd_projection_outlyingness_sorted_f64_dev(sd_ctx *ctx, const double *d_sorted, int64_t nS, int64_t T,
                                              const double *dF_new, int64_t nY, int d, const double *U, int64_t K,
                                              double *d_o_out) {
    return sorted_query_call(ctx, d_sorted, nS, T, dF_new, nY, nY, d, U, K, PJ_OUTLYING, d_o_out,
                             "sd_projection_outlyingness_sorted_f64_dev");
}

int sd_band_halfspace_sorted_f64_dev(sd_ctx *ctx, const double *d_sorted, int64_t T, int64_t nS, const double *dY,
                                     int64_t nY, int64_t ldY, int64_t *d_count_out) {
    return sorted_query_call(ctx, d_sorted, nS, T, dY, nY, ldY, 1, nullptr, 1, PJ_TUKEY, d_count_out,
                             "sd_band_halfspace_sorted_f64_dev");
}

int sd_band_outlyingness_sorted_f64_dev(sd_ctx *ctx, const double *d_sorted, int64_t T, int64_t nS,
                                        const double *dY, int64_t nY, int64_t ldY, double *d_o_out) {
    return sorted_query_call(ctx, d_sorted, nS, T, dY, nY, ldY, 1, nullptr, 1, PJ_OUTLYING, d_o_out,
                             "sd_band_outlyingness_sorted_f64_dev");
}

// ---------------------------------------------------------------------------------------------
// functional spatial depth (K14, spatial.cu)
// ---------------------------------------------------------------------------------------------
int sd_spatial_norms_f64(sd_ctx *ctx, const double *X, int64_t n, int64_t F, int layout, const int64_t *query_idx,
                         int64_t nq, double *r_out) {
    const char *who = "sd_spatial_norms_f64";
    SD_REQUIRE(n >= 1 && F >= 1 && nq >= 0, "%s: bad sizes n=%lld F=%lld nq=%lld", who, (long long)n, (long long)F,
               (long long)nq);
    SD_REQUIRE(layout == SD_LAYOUT_TN || layout == SD_LAYOUT_NT, "%s: bad layout %d", who, layout);
    SD_REQUIRE(query_idx || nq == n, "%s: query_idx == NULL requires nq == n", who);
    const double *dX = nullptr;
    const i64 *d_q = nullptr;
    double *d_r = nullptr;
    return call(ctx, who, X, r_out, true, [&](Staging &s) -> int {
        SD_TRY(upload_curves(s, X, n, nullptr, 0, F, layout, &dX));
        SD_TRY(upload_queries(ctx, query_idx, nq, n, &d_q, who));
        return s.output(BUF_OUT, r_out, nq, &d_r);
    }, [&]() -> int {
        SD_TRY(finite_check_device(ctx, dX, 1, n * F, n * F));
        return spatial_device(ctx, dX, d_q, nq, dX, n, F, d_r);
    });
}

static int spatial_of_call(sd_ctx *ctx, const double *S, i64 nS, const double *Y, i64 nY, i64 F, int layout,
                           double *r, bool dev, const char *who) {
    SD_REQUIRE(Y || nY == 0, "%s: NULL Y", who);
    SD_REQUIRE(nS >= 1 && nY >= 0 && F >= 1, "%s: bad sizes nS=%lld nY=%lld F=%lld", who, (long long)nS,
               (long long)nY, (long long)F);
    SD_REQUIRE(layout == SD_LAYOUT_TN || layout == SD_LAYOUT_NT, "%s: bad layout %d", who, layout);
    const double *dS = S, *dY = Y;
    double *d_r = r;
    return call(ctx, who, S, r, !dev, [&](Staging &s) -> int {
        if (dev) return SD_OK;
        const double *dP = nullptr;
        SD_TRY(upload_curves(s, S, nS, Y, nY, F, layout, &dP));
        dS = dP;
        dY = dP + nS * F;
        return s.output(BUF_OUT, r, nY, &d_r);
    }, [&]() -> int {
        SD_TRY(finite_check_device(ctx, dS, 1, nS * F, nS * F));
        SD_TRY(finite_check_device(ctx, dY, 1, nY * F, nY * F));
        return spatial_device(ctx, dY, nullptr, nY, dS, nS, F, d_r);
    });
}

int sd_spatial_norms_of_f64(sd_ctx *ctx, const double *S, int64_t nS, const double *Y, int64_t nY, int64_t F,
                            int layout, double *r_out) {
    return spatial_of_call(ctx, S, nS, Y, nY, F, layout, r_out, false, "sd_spatial_norms_of_f64");
}

int sd_spatial_norms_of_f64_dev(sd_ctx *ctx, const double *dS, int64_t nS, const double *dY, int64_t nY, int64_t F,
                                double *d_r_out) {
    return spatial_of_call(ctx, dS, nS, dY, nY, F, SD_LAYOUT_NT, d_r_out, true, "sd_spatial_norms_of_f64_dev");
}

}  // extern "C"
