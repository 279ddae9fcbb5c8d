// ctx.cu -- context, workspace, error and timing plumbing of libsdepth.so.
#include <stdarg.h>

#include <new>

#include "common.cuh"

namespace sd {

static thread_local char g_err[512] = "";

void set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int DevBuf::reserve(size_t bytes) {
    if (bytes <= cap) return SD_OK;
    if (p) {
        cudaFree(p);
        p = nullptr;
        cap = 0;
    }
    // round up so that repeated slightly-growing requests do not reallocate every time
    size_t want = (bytes + (1u << 20) - 1) & ~((size_t)(1u << 20) - 1);
    cudaError_t e = cudaMalloc(&p, want);
    if (e != cudaSuccess) {
        p = nullptr;
        set_error("cudaMalloc(%zu bytes) failed: %s", want, cudaGetErrorString(e));
        return SD_ERR_CUDA;
    }
    cap = want;
    return SD_OK;
}

void DevBuf::release() {
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
}

int begin_call(sd_ctx *ctx) {
    SD_CUDA(cudaSetDevice(ctx->device));
    if (ctx->pending) {  // an asynchronous call is still open: complete it (its events are about to be reused)
        ctx->pending = 0;
        SD_TRY(end_call(ctx, false));
    }
    ctx->last = sd_timings{0, 0, 0, 0, 0, 0};
    ctx->prof_n = 0;
    for (int i = 0; i < SD_PHASE_COUNT; ++i) ctx->phase_ns[i] = 0;
    SD_CUDA(cudaMemsetAsync(ctx->d_status, 0, 4 * sizeof(int), ctx->stream));
    SD_CUDA(cudaEventRecord(ctx->ev[0], ctx->stream));
    return SD_OK;
}

int prof_begin(sd_ctx *ctx, int phase) {
    if (!ctx->profile || ctx->prof_n >= sd_ctx::MAX_PROF) return SD_OK;
    const int i = ctx->prof_n;
    for (int k = 0; k < 2; ++k)
        if (!ctx->prof_ev[2 * i + k]) SD_CUDA(cudaEventCreate(&ctx->prof_ev[2 * i + k]));
    ctx->prof_phase[i] = phase;
    SD_CUDA(cudaEventRecord(ctx->prof_ev[2 * i], ctx->stream));
    return SD_OK;
}

int prof_end(sd_ctx *ctx) {
    if (!ctx->profile || ctx->prof_n >= sd_ctx::MAX_PROF) return SD_OK;
    SD_CUDA(cudaEventRecord(ctx->prof_ev[2 * ctx->prof_n + 1], ctx->stream));
    ctx->prof_n++;
    return SD_OK;
}

int mark(sd_ctx *ctx, int which) {
    SD_CUDA(cudaEventRecord(ctx->ev[which], ctx->stream));
    return SD_OK;
}

int check_status(sd_ctx *ctx) {
    const int st = *ctx->h_status;
    if (st & ST_NONFINITE) {
        set_error("input contains NaN or +-inf (the B200 engine rejects non-finite values)");
        return SD_ERR_NONFINITE;
    }
    if (st & ST_OVERFLOW) {
        set_error("a squared distance overflows float64 (differences of about 1.3e154 or more)");
        return SD_ERR_OVERFLOW;
    }
    if (st & ST_NO_MEMBER) {
        set_error("the member mask selects no curve");
        return SD_ERR_INVALID;
    }
    if (st & ST_BAD_INPUT) {
        set_error("input value out of range (extremities must lie in [0, n - 1])");
        return SD_ERR_INVALID;
    }
    if (st & ST_INTERNAL) {
        set_error("internal consistency check failed on the device (status=%d)", st);
        return SD_ERR_CUDA;
    }
    return SD_OK;
}

int end_call(sd_ctx *ctx, bool had_copies) {
    SD_CUDA(cudaMemcpyAsync(ctx->h_status, ctx->d_status, 4 * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    SD_CUDA(cudaEventRecord(ctx->ev[3], ctx->stream));
    SD_CUDA(cudaStreamSynchronize(ctx->stream));
    float ms = 0.f;
    if (had_copies) {
        SD_CUDA(cudaEventElapsedTime(&ms, ctx->ev[0], ctx->ev[1]));
        ctx->last.h2d_ns = (int64_t)(ms * 1e6);
        SD_CUDA(cudaEventElapsedTime(&ms, ctx->ev[2], ctx->ev[3]));
        ctx->last.d2h_ns = (int64_t)(ms * 1e6);
    }
    SD_CUDA(cudaEventElapsedTime(&ms, ctx->ev[1], ctx->ev[2]));
    ctx->last.kernel_ns = (int64_t)(ms * 1e6);
    ctx->last.fallback_rows = ctx->h_status[1];
    for (int i = 0; i < ctx->prof_n; ++i) {
        SD_CUDA(cudaEventElapsedTime(&ms, ctx->prof_ev[2 * i], ctx->prof_ev[2 * i + 1]));
        ctx->phase_ns[ctx->prof_phase[i]] += (int64_t)(ms * 1e6);
    }
    return check_status(ctx);
}

// ---------------------------------------------------------------------------------------------
// small utility kernels
// ---------------------------------------------------------------------------------------------
__global__ void transpose_kernel(const double *__restrict__ in, i64 rows, i64 cols, i64 ld_in,
                                 double *__restrict__ out) {
    __shared__ double tile[32][33];
    const i64 c0 = (i64)blockIdx.x * 32, r0 = (i64)blockIdx.y * 32;
    for (int dy = threadIdx.y; dy < 32; dy += blockDim.y) {
        const i64 r = r0 + dy, c = c0 + threadIdx.x;
        if (r < rows && c < cols) tile[dy][threadIdx.x] = in[r * ld_in + c];
    }
    __syncthreads();
    for (int dy = threadIdx.y; dy < 32; dy += blockDim.y) {
        const i64 c = c0 + dy, r = r0 + threadIdx.x;
        if (r < rows && c < cols) out[c * rows + r] = tile[threadIdx.x][dy];
    }
}

// out[cols][rows] = in[rows][cols]^T
int transpose_device(sd_ctx *ctx, const double *d_in, i64 rows, i64 cols, i64 ld_in, double *d_out) {
    if (rows == 0 || cols == 0) return SD_OK;
    dim3 grid((unsigned)ceil_div(cols, 32), (unsigned)ceil_div(rows, 32));
    dim3 block(32, 8);
    if (grid.y > 65535) {
        set_error("transpose: too many rows (%lld)", (long long)rows);
        return SD_ERR_UNSUPPORTED;
    }
    transpose_kernel<<<grid, block, 0, ctx->stream>>>(d_in, rows, cols, ld_in, d_out);
    ctx->last.launches++;
    SD_CUDA(cudaGetLastError());
    return SD_OK;
}

__global__ void gather_i64_kernel(const i64 *__restrict__ src, const i64 *__restrict__ idx, i64 nq,
                                  i64 *__restrict__ out) {
    const i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < nq) out[i] = src[idx ? idx[i] : i];
}

int gather_i64_device(sd_ctx *ctx, const i64 *d_src, const i64 *d_idx, i64 nq, i64 *d_out) {
    if (nq == 0) return SD_OK;
    gather_i64_kernel<<<(unsigned)ceil_div(nq, 256), 256, 0, ctx->stream>>>(d_src, d_idx, nq, d_out);
    ctx->last.launches++;
    SD_CUDA(cudaGetLastError());
    return SD_OK;
}

// out[(b*T + t)*m + k] = X[t*n + cols[b*m + k]] for nb batches of m member columns each
__global__ void compact_batches_kernel(const double *__restrict__ X, i64 T, i64 n, const i64 *__restrict__ cols,
                                       i64 m, i64 nb, double *__restrict__ out) {
    const i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nb * T * m) return;
    const i64 k = i % m, bt = i / m;
    const i64 t = bt % T, b = bt / T;
    out[i] = X[t * n + cols[b * m + k]];
}

int compact_batches_device(sd_ctx *ctx, const double *dX, i64 T, i64 n, const i64 *d_cols, i64 m, i64 nb,
                           double *d_out) {
    if (nb * T * m == 0) return SD_OK;
    compact_batches_kernel<<<(unsigned)ceil_div(nb * T * m, 256), 256, 0, ctx->stream>>>(dX, T, n, d_cols, m, nb,
                                                                                          d_out);
    ctx->last.launches++;
    SD_CUDA(cudaGetLastError());
    return SD_OK;
}

// out[t*m + k] = X[t*n + cols[k]]
__global__ void compact_columns_kernel(const double *__restrict__ X, i64 T, i64 n, const i64 *__restrict__ cols,
                                       i64 m, double *__restrict__ out) {
    const i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= T * m) return;
    const i64 t = i / m, k = i - t * m;
    out[i] = X[t * n + cols[k]];
}

int compact_columns_device(sd_ctx *ctx, const double *dX, i64 T, i64 n, const i64 *d_cols, i64 m, double *d_out) {
    if (T * m == 0) return SD_OK;
    compact_columns_kernel<<<(unsigned)ceil_div(T * m, 256), 256, 0, ctx->stream>>>(dX, T, n, d_cols, m, d_out);
    ctx->last.launches++;
    SD_CUDA(cudaGetLastError());
    return SD_OK;
}

}  // namespace sd

// ---------------------------------------------------------------------------------------------
// C ABI: context management
// ---------------------------------------------------------------------------------------------
extern "C" {

int sd_abi_version(void) { return SD_ABI_VERSION; }

const char *sd_last_error(void) { return sd::g_err; }

int sd_init(int device, sd_ctx **out) {
    if (!out) {
        sd::set_error("sd_init: out is NULL");
        return SD_ERR_INVALID;
    }
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) {
        sd::set_error("sd_init: no CUDA device (%s)", e == cudaSuccess ? "count == 0" : cudaGetErrorString(e));
        return SD_ERR_NO_DEVICE;
    }
    if (device < 0 || device >= count) {
        sd::set_error("sd_init: device %d out of range [0,%d)", device, count);
        return SD_ERR_INVALID;
    }
    cudaDeviceProp prop;
    SD_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) {
        sd::set_error("sd_init: device %d is sm_%d%d; this library is built for sm_100a (B200) only", device,
                      prop.major, prop.minor);
        return SD_ERR_NO_DEVICE;
    }
    SD_CUDA(cudaSetDevice(device));
    sd_ctx *ctx = new (std::nothrow) sd_ctx();
    if (!ctx) {
        sd::set_error("sd_init: out of host memory");
        return SD_ERR_INVALID;
    }
    ctx->device = device;
    ctx->sm_count = prop.multiProcessorCount;
    SD_CUDA(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
    SD_CUDA(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
    for (int i = 0; i < 4; ++i) SD_CUDA(cudaEventCreateWithFlags(&ctx->ev_pipe[i], cudaEventDisableTiming));
    for (int i = 0; i < 4; ++i) SD_CUDA(cudaEventCreate(&ctx->ev[i]));
    SD_CUDA(cudaMalloc(&ctx->d_status, 8 * sizeof(int)));
    SD_CUDA(cudaMemset(ctx->d_status, 0, 8 * sizeof(int)));  // [6..7]: the slab path's counters, left at zero by every call
    SD_CUDA(cudaHostAlloc(&ctx->h_status, 4 * sizeof(int), cudaHostAllocMapped));
    SD_CUDA(cudaHostGetDevicePointer(&ctx->h_status_dev, ctx->h_status, 0));
    memset(ctx->h_status, 0, 4 * sizeof(int));
    *out = ctx;
    return SD_OK;
}

int sd_destroy(sd_ctx *ctx) {
    if (!ctx) return SD_OK;
    cudaSetDevice(ctx->device);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    for (int i = 0; i < sd::NUM_BUFS; ++i) ctx->buf[i].release();
    if (ctx->d_status) cudaFree(ctx->d_status);
    if (ctx->h_status) cudaFreeHost(ctx->h_status);
    for (int i = 0; i < 4; ++i)
        if (ctx->ev[i]) cudaEventDestroy(ctx->ev[i]);
    for (int i = 0; i < 2 * sd_ctx::MAX_PROF; ++i)
        if (ctx->prof_ev[i]) cudaEventDestroy(ctx->prof_ev[i]);
    for (int i = 0; i < 4; ++i)
        if (ctx->ev_pipe[i]) cudaEventDestroy(ctx->ev_pipe[i]);
    for (int i = 0; i < 2; ++i) {
        if (ctx->ev_stage[i]) cudaEventDestroy(ctx->ev_stage[i]);
        if (ctx->stage[i]) cudaFreeHost(ctx->stage[i]);
    }
    for (int i = 0; i < 2; ++i)
        if (ctx->ev_slab[i]) cudaEventDestroy(ctx->ev_slab[i]);
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
    return SD_OK;
}

int sd_device_info(sd_ctx *ctx, sd_devinfo *out) {
    if (!ctx || !out) {
        sd::set_error("sd_device_info: NULL argument");
        return SD_ERR_INVALID;
    }
    cudaDeviceProp prop;
    SD_CUDA(cudaGetDeviceProperties(&prop, ctx->device));
    out->device = ctx->device;
    out->sm_count = prop.multiProcessorCount;
    out->cc_major = prop.major;
    out->cc_minor = prop.minor;
    out->total_mem = (int64_t)prop.totalGlobalMem;
    strncpy(out->name, prop.name, sizeof(out->name) - 1);
    out->name[sizeof(out->name) - 1] = 0;
    return SD_OK;
}

int sd_set_option(sd_ctx *ctx, int option, int64_t value) {
    if (!ctx) {
        sd::set_error("sd_set_option: NULL context");
        return SD_ERR_INVALID;
    }
    switch (option) {
        case SD_OPT_BD_IMPL:
            if (value < SD_BD_AUTO || value > SD_BD_MATCH) {
                sd::set_error("sd_set_option: bad SD_OPT_BD_IMPL value %lld", (long long)value);
                return SD_ERR_INVALID;
            }
            ctx->bd_impl = (int)value;
            return SD_OK;
        case SD_OPT_MBD_FORCE_FALLBACK:
            ctx->mbd_force_fallback = value ? 1 : 0;
            return SD_OK;
        case SD_OPT_PROFILE:
            ctx->profile = value ? 1 : 0;
            return SD_OK;
        case SD_OPT_SIMPLICIAL_IMPL:
            if (value < SD_SIMPLICIAL_AUTO || value > SD_SIMPLICIAL_COUNT) {
                sd::set_error("sd_set_option: bad SD_OPT_SIMPLICIAL_IMPL value %lld", (long long)value);
                return SD_ERR_INVALID;
            }
            ctx->simplicial_impl = (int)value;
            return SD_OK;
        case SD_OPT_ASYNC_DEVICE:
            ctx->async_device = value ? 1 : 0;
            return SD_OK;
        default:
            sd::set_error("sd_set_option: unknown option %d", option);
            return SD_ERR_INVALID;
    }
}

int sd_get_timings(sd_ctx *ctx, sd_timings *out) {
    if (!ctx || !out) {
        sd::set_error("sd_get_timings: NULL argument");
        return SD_ERR_INVALID;
    }
    *out = ctx->last;
    return SD_OK;
}

int sd_get_phase_ns(sd_ctx *ctx, int64_t *out) {
    if (!ctx || !out) {
        sd::set_error("sd_get_phase_ns: NULL argument");
        return SD_ERR_INVALID;
    }
    for (int i = 0; i < SD_PHASE_COUNT; ++i) out[i] = ctx->phase_ns[i];
    return SD_OK;
}

int sd_probe_int8_peak(sd_ctx *ctx, double *ops_per_s) {
    if (!ctx || !ops_per_s) {
        sd::set_error("sd_probe_int8_peak: NULL argument");
        return SD_ERR_INVALID;
    }
    SD_CUDA(cudaSetDevice(ctx->device));
    return sd::probe_int8_peak(ctx, ops_per_s);
}

void *sd_stream(sd_ctx *ctx) { return ctx ? (void *)ctx->stream : nullptr; }

int sd_sync(sd_ctx *ctx) {
    if (!ctx) {
        sd::set_error("sd_sync: NULL context");
        return SD_ERR_INVALID;
    }
    SD_CUDA(cudaSetDevice(ctx->device));
    if (ctx->pending) {
        ctx->pending = 0;
        return sd::end_call(ctx, false);
    }
    SD_CUDA(cudaStreamSynchronize(ctx->stream));
    return SD_OK;
}

}  // extern "C"
