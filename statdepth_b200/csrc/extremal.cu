// extremal.cu -- extremal depth (Narisetty & Nair 2016): curves ordered by the left tail of their pointwise-depth
// distribution (K10).
//
// With b_t(c) / a_t(c) the other curves strictly below / above curve c at row t (the integers K1 ranks with), the
// pointwise extremity is m_t(c) = |b_t(c) - a_t(c)| in [0, n - 1] (the paper's pointwise depth is 1 - m / n).  The
// key of curve c is its T extremities sorted descending; keys compare lexicographically, a larger key being more
// extreme (the first depth level at which two depth CDFs differ decides, and that is the first differing key
// element).  The numerator e(c) = #{h : key(h) >= key(c)} in [1, n]; ED = e / n, the deepest curve has e = n.
//
// Stage 1 (extremity_device): rank-only passes of the rank pipeline in row blocks (for_each_rank_block, mbd.cu);
//   extremity_kernel writes m[t*n + c] as int32, row-major.  A rank outside 0 <= b, a, b + a <= n - 1 sets
//   ST_INTERNAL (never a trap); the finite check is K1's.  Rows are independent, so a block of time rows gives those
//   rows of m (the multi-GPU split).
// Stage 2a (extremal_keys_kernel): one CTA per group of G consecutive curves.  It reads rows of m coalesced along c,
//   places curve g's T values in segment g (2^ceil(log2 T) slots, padded with 0, which sorts last) of a shared tile,
//   sorts every segment descending with one segmented bitonic network (compare-exchanges never cross a segment),
//   and writes keys[c*T + 0..T) as u32, curve-major.  The tile is KEY_TILE slots at small T (G = KEY_TILE / seg, so
//   T = 1, n = 10^7 launches 1221 CTAs, not 10^7), one segment above; T <= KEY_T_MAX keeps one segment within the
//   64 KB of dynamic shared memory the kernel is given.  An m value outside [0, n - 1] sets ST_BAD_INPUT.
// Stage 2b: cub::DeviceMergeSort sorts the curve ids by key ascending (least extreme first) with a lexicographic
//   comparator over keys; group_starts_kernel marks p where key(ids[p - 1]) != key(ids[p]) with p (else 0), an
//   inclusive max-scan (cub::DeviceScan) carries each group's start s over the group, and scatter_kernel writes
//   e[ids[p]] = n - s in int64.  Equal keys are one group, so they get equal e.
// Buffers: stage 1 holds BUF_RANKS and the rank pipeline's buffers; stage 2 uses only BUF_KEYS and BUF_ORDER, so it
// can follow stage 1 or the boxplot's envelope pass (BUF_AUX) on the same stream without touching what they hold.
#define CCCL_DISABLE_NVTX
#include <cub/device/device_merge_sort.cuh>
#include <cub/device/device_scan.cuh>

#include "common.cuh"

namespace sd {

constexpr int EXT_THREADS = 256;
constexpr i64 EXT_MAX_ROWS = 65535;  // row block cap, as the other rank-only drivers
constexpr int KEY_THREADS = 512;
constexpr int KEY_TILE = 8192;  // u32 slots of a CTA's tile at T <= KEY_TILE (32 KB)
static_assert(SD_EXTREMAL_T_MAX * 4 <= 64 * 1024, "one key segment must fit the kernel's 64 KB of shared memory");
constexpr int ORDER_THREADS = 256;

__global__ void __launch_bounds__(EXT_THREADS) extremity_kernel(const int *__restrict__ rb, const int *__restrict__ ra,
                                                                const i64 n, const i64 count, int *__restrict__ m,
                                                                int *__restrict__ status) {
    bool bad = false;
    for (i64 i = (i64)blockIdx.x * EXT_THREADS + threadIdx.x; i < count; i += (i64)gridDim.x * EXT_THREADS) {
        const int b = rb[i], a = ra[i];
        bad |= b < 0 || a < 0 || (i64)b + a > n - 1;
        m[i] = b > a ? b - a : a - b;
    }
    if (bad) atomicOr(status, ST_INTERNAL);
}

int extremity_device(sd_ctx *ctx, const double *dX, i64 T, i64 n, i64 ld, int *d_m) {
    if (T < 1 || n < 1 || ld < n) {
        set_error("band extremity: bad shape T=%lld n=%lld ld=%lld", (long long)T, (long long)n, (long long)ld);
        return SD_ERR_INVALID;
    }
    cudaStream_t st = ctx->stream;
    return for_each_rank_block(ctx, dX, T, n, ld, true, EXT_MAX_ROWS,
                               [&](i64 r0, i64 rows, const int *rb, const int *ra) {
        i64 grid = ceil_div(rows * n, EXT_THREADS);
        if (grid > 8 * (i64)ctx->sm_count) grid = 8 * (i64)ctx->sm_count;
        extremity_kernel<<<(unsigned)grid, EXT_THREADS, 0, st>>>(rb, ra, n, rows * n, d_m + r0 * n, ctx->d_status);
        ctx->last.launches++;
    });
}

// grid: one CTA per G = tile >> seg_log curves; dynamic shared memory: tile u32
__global__ void __launch_bounds__(KEY_THREADS) extremal_keys_kernel(const int *__restrict__ m, const int T,
                                                                    const i64 n, const int seg_log, const int tile,
                                                                    u32 *__restrict__ keys,
                                                                    int *__restrict__ status) {
    extern __shared__ u32 s[];
    const int seg = 1 << seg_log, G = tile >> seg_log;
    const i64 c0 = (i64)blockIdx.x * G;
    const int here = n - c0 < G ? (int)(n - c0) : G;
    bool bad = false;
    for (int idx = threadIdx.x; idx < tile; idx += KEY_THREADS) {  // consecutive threads: consecutive curves
        const int g = idx & (G - 1), t = idx >> (31 - __clz(G));
        u32 v = 0;
        if (t < T && g < here) {
            const int x = m[(i64)t * n + c0 + g];
            if (x < 0 || x >= n) bad = true;
            else v = (u32)x;
        }
        s[(g << seg_log) + t] = v;
    }
    if (bad) atomicOr(status, ST_BAD_INPUT);
    __syncthreads();
    // bitonic network, descending within every segment: at k == seg every block is descending, before that the
    // blocks alternate so that each merge sees a bitonic sequence
    for (int k = 2; k <= seg; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int p = threadIdx.x; p < (tile >> 1); p += KEY_THREADS) {
                const int lo = ((p & ~(j - 1)) << 1) | (p & (j - 1));  // p with a 0 inserted at bit log2(j)
                const int hi = lo | j;
                const u32 a = s[lo], b = s[hi];
                const bool desc = (lo & (seg - 1) & k) == 0;
                if (desc ? a < b : a > b) {
                    s[lo] = b;
                    s[hi] = a;
                }
            }
            __syncthreads();
        }
    }
    u32 *out = keys + c0 * T;
    for (int idx = threadIdx.x; idx < here * T; idx += KEY_THREADS) {
        const int g = idx / T, t = idx - g * T;
        out[idx] = s[(g << seg_log) + t];
    }
}

struct KeyLess {
    const u32 *keys;
    i64 T;
    __device__ __forceinline__ bool operator()(const int a, const int b) const {
        const u32 *ka = keys + (i64)a * T, *kb = keys + (i64)b * T;
        for (i64 i = 0; i < T; ++i) {
            const u32 x = ka[i], y = kb[i];
            if (x != y) return x < y;
        }
        return false;
    }
};

struct MaxOp {
    __device__ __forceinline__ int operator()(const int a, const int b) const { return a > b ? a : b; }
};

__global__ void group_starts_kernel(const int *__restrict__ ids, const u32 *__restrict__ keys, const i64 T,
                                    const i64 n, int *__restrict__ start) {
    const i64 p = (i64)blockIdx.x * ORDER_THREADS + threadIdx.x;
    if (p >= n) return;
    bool first = p == 0;
    if (!first) {
        const u32 *ka = keys + (i64)ids[p - 1] * T, *kb = keys + (i64)ids[p] * T;
        for (i64 i = 0; i < T && !first; ++i) first = ka[i] != kb[i];
    }
    start[p] = first ? (int)p : 0;
}

__global__ void ids_kernel(int *__restrict__ ids, const i64 n) {
    const i64 p = (i64)blockIdx.x * ORDER_THREADS + threadIdx.x;
    if (p < n) ids[p] = (int)p;
}

__global__ void scatter_kernel(const int *__restrict__ ids, const int *__restrict__ start, const i64 n,
                               i64 *__restrict__ e) {
    const i64 p = (i64)blockIdx.x * ORDER_THREADS + threadIdx.x;
    if (p < n) e[ids[p]] = n - start[p];
}

static size_t align256(size_t b) { return (b + 255) & ~(size_t)255; }

int extremal_depth_device(sd_ctx *ctx, const int *d_m, i64 T, i64 n, i64 *d_e) {
    if (T < 1 || n < 1 || n > 0x7fffffffll) {
        set_error("extremal depth: bad shape T=%lld n=%lld", (long long)T, (long long)n);
        return SD_ERR_INVALID;
    }
    if (T > SD_EXTREMAL_T_MAX) {
        set_error("extremal depth: T=%lld time points exceed the per-curve sort's bound of %d", (long long)T,
                  SD_EXTREMAL_T_MAX);
        return SD_ERR_INVALID;
    }
    cudaStream_t st = ctx->stream;
    int seg_log = 0;
    while ((1ll << seg_log) < T) ++seg_log;
    const int tile = (1 << seg_log) > KEY_TILE ? (1 << seg_log) : KEY_TILE;
    const i64 G = tile >> seg_log;
    SD_TRY(ctx->buf[BUF_KEYS].reserve((size_t)T * n * sizeof(u32)));
    u32 *keys = ctx->buf[BUF_KEYS].as<u32>();
    const size_t smem = (size_t)tile * sizeof(u32);
    SD_CUDA(cudaFuncSetAttribute(extremal_keys_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    extremal_keys_kernel<<<(unsigned)ceil_div(n, G), KEY_THREADS, smem, st>>>(d_m, (int)T, n, seg_log, tile, keys,
                                                                                ctx->d_status);
    ctx->last.launches++;
    SD_CUDA(cudaGetLastError());

    // BUF_ORDER: ids [n] | start [n] | scanned start [n] | cub temp storage (merge sort, then the scan)
    const int N = (int)n;
    const KeyLess less{keys, T};
    size_t sort_bytes = 0, scan_bytes = 0;
    SD_CUDA(cub::DeviceMergeSort::SortKeys(nullptr, sort_bytes, (int *)nullptr, N, less, st));
    SD_CUDA(cub::DeviceScan::InclusiveScan(nullptr, scan_bytes, (const int *)nullptr, (int *)nullptr, MaxOp{}, N, st));
    const size_t vec = align256((size_t)n * sizeof(int));
    const size_t temp = sort_bytes > scan_bytes ? sort_bytes : scan_bytes;
    SD_TRY(ctx->buf[BUF_ORDER].reserve(3 * vec + temp));
    char *base = ctx->buf[BUF_ORDER].as<char>();
    int *ids = reinterpret_cast<int *>(base), *start = reinterpret_cast<int *>(base + vec);
    int *scanned = reinterpret_cast<int *>(base + 2 * vec);
    void *d_temp = base + 3 * vec;
    const unsigned grid = (unsigned)ceil_div(n, ORDER_THREADS);
    ids_kernel<<<grid, ORDER_THREADS, 0, st>>>(ids, n);
    ctx->last.launches++;
    SD_CUDA(cudaGetLastError());
    SD_CUDA(cub::DeviceMergeSort::SortKeys(d_temp, sort_bytes, ids, N, less, st));
    ctx->last.launches++;
    group_starts_kernel<<<grid, ORDER_THREADS, 0, st>>>(ids, keys, T, n, start);
    ctx->last.launches++;
    SD_CUDA(cudaGetLastError());
    SD_CUDA(cub::DeviceScan::InclusiveScan(d_temp, scan_bytes, start, scanned, MaxOp{}, N, st));
    ctx->last.launches++;
    scatter_kernel<<<grid, ORDER_THREADS, 0, st>>>(ids, scanned, n, d_e);
    ctx->last.launches++;
    SD_CUDA(cudaGetLastError());
    return SD_OK;
}

}  // namespace sd
