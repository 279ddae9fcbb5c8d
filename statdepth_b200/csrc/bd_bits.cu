// bd_bits.cu -- strict band depth (relax=False) as bit-packed sign masks + early-exit pair tests.
//
// Replaces the strict branch of _r2_containment (_containment.py:68-80: containment // len(curve))
// enumerated over all pairs by _univariate_band_depth (_functional.py:238-253).  For query curve q
//     Sb[c][t] = [X[t,c] < X[t,q]],  Sa[c][t] = [X[t,c] > X[t,q]]
// and a pair (c1 < c2) of OTHER curves contains q at every time point iff
//     (Sb[c1] & Sb[c2]) | (Sa[c1] & Sa[c2]) == 0      over all T bits
// i.e. iff the violation Gram entry V[c1,c2] = Sb.Sb^T + Sa.Sa^T is zero (SURVEY 8a row a3, "K2").
// This file is the CUDA-core variant: masks are packed 32 time points per word, word-major so the
// first word of every curve (which rejects ~99 % of pairs of crossing curves) is contiguous, and are
// stored for the n-1 OTHER curves only (position o = c - [c > q]) so the pair loop carries no index
// tests.  Every thread keeps the first word of 4 curves in registers and streams the partners' first
// words from shared memory (1 LDS + 8 LOP3 per 4 pairs); survivors are queued in shared memory and
// verified on the remaining words by the whole CTA.
// The tcgen05 int8 Gram variant lives in bd_gemm.cu; sd_set_option(SD_OPT_BD_IMPL) selects.
#include "common.cuh"

namespace sd {

constexpr int MASK_QT = 8;       // queries handled per thread by the mask kernel
constexpr int PAIR_THREADS = 256;
constexpr int PAIR_JPT = 4;      // curves per thread
constexpr int PAIR_TJ = PAIR_THREADS * PAIR_JPT;  // 1024 curves per J tile
constexpr int PAIR_TK = 512;     // partner curves staged per K tile
constexpr int PAIR_QCAP = 4096;

// M[(q*W + w)*m + o] = {below bits, above bits} of other curve o vs query q (m = n - 1 others; curve id
// c = o + [o >= q]).  Bit b of word w is time point t = w + W*b: every word SPANS the whole time axis, so
// word 0 already samples 32 widely spaced time points.  (With 32 consecutive time points per word, sign
// persistence of smooth curves let ~5 % of all pairs survive word 0 and the verification of survivors
// dominated the kernel.)
__global__ void __launch_bounds__(128) bd_mask_kernel(const double *__restrict__ X, const i64 T, const i64 n,
                                                      const i64 ld, const i64 *__restrict__ qidx, const int nqb,
                                                      const int W, uint2 *__restrict__ M,
                                                      int *__restrict__ status) {
    __shared__ double sq[32][MASK_QT];
    __shared__ i64 sqi[MASK_QT];
    const int w = blockIdx.y;
    const int q0 = blockIdx.z * MASK_QT;
    if (threadIdx.x < MASK_QT) sqi[threadIdx.x] = q0 + threadIdx.x < nqb ? qidx[q0 + threadIdx.x] : 0;
    for (int i = threadIdx.x; i < 32 * MASK_QT; i += blockDim.x) {
        const int tt = i / MASK_QT, qq = i % MASK_QT;
        const i64 t = (i64)w + (i64)W * tt;
        double v = 0.0;
        if (t < T && q0 + qq < nqb) v = X[t * ld + qidx[q0 + qq]];
        sq[tt][qq] = v;
    }
    __syncthreads();
    const i64 m = n - 1;
    const i64 o = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (o >= m) return;
    u32 b[MASK_QT], a[MASK_QT];
    bool shift[MASK_QT];  // other o is curve o+1 for queries at or before o
#pragma unroll
    for (int qq = 0; qq < MASK_QT; ++qq) {
        b[qq] = a[qq] = 0u;
        shift[qq] = o >= sqi[qq];
    }
    bool bad = false;
    for (int tt = 0; tt < 32; ++tt) {
        const i64 t = (i64)w + (i64)W * tt;
        if (t >= T) break;
        const double *row = X + t * ld;
        const double x0 = row[o], x1 = row[o + 1];  // o + 1 <= n - 1
        bad |= !isfinite(x0) || !isfinite(x1);
#pragma unroll
        for (int qq = 0; qq < MASK_QT; ++qq) {
            const double x = shift[qq] ? x1 : x0;
            const double xq = sq[tt][qq];
            b[qq] |= (u32)(x < xq) << tt;
            a[qq] |= (u32)(x > xq) << tt;
        }
    }
    if (bad) atomicOr(status, ST_NONFINITE);
#pragma unroll
    for (int qq = 0; qq < MASK_QT; ++qq)
        if (q0 + qq < nqb) M[((i64)(q0 + qq) * W + w) * m + o] = make_uint2(b[qq], a[qq]);
}

__device__ __forceinline__ bool pair_survives_tail(const uint2 *__restrict__ Mq, const int W, const i64 m, const int o1,
                                                   const int o2) {
    for (int w = 1; w < W; ++w) {
        const uint2 m1 = Mq[(i64)w * m + o1], m2 = Mq[(i64)w * m + o2];
        if ((m1.x & m2.x) | (m1.y & m2.y)) return false;
    }
    return true;
}

struct PairQueue {
    uint2 *items;
    int *count;
};

// a pair passed word 0: count it (W == 1) or queue it for the remaining words
__device__ __forceinline__ void pair_hit(const PairQueue &pq, const uint2 *__restrict__ Mq, const int W, const i64 m,
                                         const int o1, const int o2, u64 &count) {
    if (W == 1) {
        ++count;
        return;
    }
    const int pos = atomicAdd(pq.count, 1);
    if (pos < PAIR_QCAP) pq.items[pos] = make_uint2((u32)o1, (u32)o2);
    else count += pair_survives_tail(Mq, W, m, o1, o2);  // queue full: verify in place
}

__device__ __forceinline__ void pair_drain(const PairQueue &pq, const uint2 *__restrict__ Mq, const int W, const i64 m,
                                           u64 &count) {
    __syncthreads();
    const int qn = *pq.count < PAIR_QCAP ? *pq.count : PAIR_QCAP;
    for (int i = threadIdx.x; i < qn; i += PAIR_THREADS) {
        const uint2 pr = pq.items[i];
        count += pair_survives_tail(Mq, W, m, (int)pr.x, (int)pr.y);
    }
    __syncthreads();
    if (threadIdx.x == 0) *pq.count = 0;
    __syncthreads();
}

// grid (J tiles, queries).  CTA (jt, q): others o1 in J tile jt against every o2 > o1.
__global__ void __launch_bounds__(PAIR_THREADS) bd_pair_kernel(const uint2 *__restrict__ M, const i64 m, const int W,
                                                               i64 *__restrict__ out, u64 *__restrict__ hits) {
    __shared__ uint2 s_tile[PAIR_TK];
    __shared__ uint2 s_queue[PAIR_QCAP];
    __shared__ int s_qn;
    __shared__ u64 s_total;
    const int q = blockIdx.y, jt = blockIdx.x;
    const uint2 *Mq = M + (i64)q * W * m;
    const PairQueue pq = {s_queue, &s_qn};
    const i64 j0 = (i64)jt * PAIR_TJ;
    int o1[PAIR_JPT];
    uint2 m1[PAIR_JPT];
    bool ok1[PAIR_JPT];
#pragma unroll
    for (int u = 0; u < PAIR_JPT; ++u) {
        o1[u] = (int)(j0 + u * PAIR_THREADS + threadIdx.x);
        ok1[u] = o1[u] < m;
        // rows past the end get all-ones masks and are additionally guarded by ok1 where a zero can appear
        m1[u] = ok1[u] ? Mq[o1[u]] : make_uint2(0xffffffffu, 0xffffffffu);
    }
    if (threadIdx.x == 0) { s_qn = 0; s_total = 0ull; }
    u64 count = 0;
    u32 nhit = 0;  // pairs that passed word 0 (statistics for SD_BD_AUTO)
    const i64 jend = j0 + PAIR_TJ < m ? j0 + PAIR_TJ : m;  // partners below jend may have o2 <= o1
    for (i64 k0 = j0; k0 < m; k0 += PAIR_TK) {
        __syncthreads();
        const int klen = (m - k0) < PAIR_TK ? (int)(m - k0) : PAIR_TK;
        for (int i = threadIdx.x; i < klen; i += PAIR_THREADS) s_tile[i] = Mq[k0 + i];
        __syncthreads();
        const bool diag = k0 < jend;  // uniform per tile
        for (int kk = 0; kk < klen; ++kk) {
            const uint2 m2 = s_tile[kk];
            u32 v[PAIR_JPT];
#pragma unroll
            for (int u = 0; u < PAIR_JPT; ++u) v[u] = (m1[u].x & m2.x) | (m1[u].y & m2.y);
            if (!(v[0] && v[1] && v[2] && v[3])) {  // rare: some pair of this row passed word 0
                const int o2 = (int)(k0 + kk);
#pragma unroll
                for (int u = 0; u < PAIR_JPT; ++u)
                    if (v[u] == 0u && ok1[u] && (!diag || o2 > o1[u])) {
                        ++nhit;
                        pair_hit(pq, Mq, W, m, o1[u], o2, count);
                    }
            }
        }
        if (W > 1) {
            __syncthreads();
            const bool full = s_qn >= PAIR_QCAP / 2;
            __syncthreads();  // every thread has read the same s_qn before anyone pushes again
            if (full) pair_drain(pq, Mq, W, m, count);
        }
    }
    if (W > 1) pair_drain(pq, Mq, W, m, count);
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) count += __shfl_xor_sync(0xffffffffu, count, s);
    if ((threadIdx.x & 31) == 0 && count) atomicAdd(&s_total, count);
    __syncthreads();
    if (threadIdx.x == 0 && s_total) atomicAdd((u64 *)&out[q], s_total);
    if (hits) {
#pragma unroll
        for (int s = 16; s > 0; s >>= 1) nhit += __shfl_xor_sync(0xffffffffu, nhit, s);
        if ((threadIdx.x & 31) == 0 && nhit) atomicAdd(hits, (u64)nhit);
    }
}

// J = 3, strict: triples (o1 < o2 < o3) of other curves never all-below / all-above.  O(n^3 W)
// per query: meant for the small n the reference itself can handle.  One thread per (o1, o2).
__global__ void __launch_bounds__(256) bd_triple_kernel(const uint2 *__restrict__ M, const i64 m, const int W,
                                                        i64 *__restrict__ out) {
    const int q = blockIdx.y;
    const uint2 *Mq = M + (i64)q * W * m;
    const i64 npairs = m * (m - 1) / 2;
    const i64 pid = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    u64 count = 0;
    if (pid < npairs) {
        // unrank pid -> (o1 < o2): o2 = largest with o2(o2-1)/2 <= pid
        i64 o2 = (i64)((1.0 + sqrt(1.0 + 8.0 * (double)pid)) * 0.5);
        while (o2 * (o2 - 1) / 2 > pid) --o2;
        while ((o2 + 1) * o2 / 2 <= pid) ++o2;
        const i64 o1 = pid - o2 * (o2 - 1) / 2;
        for (i64 o3 = o2 + 1; o3 < m; ++o3) {
            bool ok = true;
            for (int w = 0; w < W && ok; ++w) {
                const uint2 a = Mq[(i64)w * m + o1], b = Mq[(i64)w * m + o2], c = Mq[(i64)w * m + o3];
                ok = ((a.x & b.x & c.x) | (a.y & b.y & c.y)) == 0u;
            }
            count += ok;
        }
    }
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) count += __shfl_xor_sync(0xffffffffu, count, s);
    if ((threadIdx.x & 31) == 0 && count) atomicAdd((u64 *)&out[q], count);
}

// d_out[nq] receives the strict numerator for subset size j.
int bd_strict_device(sd_ctx *ctx, const double *dX, i64 T, i64 n, i64 ld, const i64 *d_q, i64 nq, int j,
                     i64 *d_out, u64 *d_hits) {
    if (n < 1 || T < 1 || ld < n || nq < 0) {
        set_error("strict band depth: bad shape T=%lld n=%lld ld=%lld nq=%lld", (long long)T, (long long)n,
                  (long long)ld, (long long)nq);
        return SD_ERR_INVALID;
    }
    if (n >= (1ll << 31)) {
        set_error("strict band depth: n=%lld exceeds 2^31-1", (long long)n);
        return SD_ERR_UNSUPPORTED;
    }
    cudaStream_t st = ctx->stream;
    SD_CUDA(cudaMemsetAsync(d_out, 0, (size_t)nq * sizeof(i64), st));
    const i64 m = n - 1;  // other curves
    if (nq == 0 || m < j) return SD_OK;
    const i64 W = ceil_div(T, 32);
    if (W > 65535) {
        set_error("strict band depth: T=%lld too large (max %d)", (long long)T, 65535 * 32);
        return SD_ERR_UNSUPPORTED;
    }
    // queries per batch: masks are W*m*8 bytes per query, keep the batch under ~2 GB
    const size_t per_q = (size_t)W * (size_t)m * sizeof(uint2);
    i64 QB = (i64)((2ull << 30) / per_q);
    if (QB < MASK_QT) QB = MASK_QT;
    if (QB > 32768) QB = 32768;
    if (QB > nq) QB = nq;
    SD_TRY(ctx->buf[BUF_MASK].reserve((size_t)QB * per_q));
    uint2 *M = ctx->buf[BUF_MASK].as<uint2>();
    for (i64 q0 = 0; q0 < nq; q0 += QB) {
        const int nqb = (int)(nq - q0 < QB ? nq - q0 : QB);
        dim3 mgrid((unsigned)ceil_div(m, 128), (unsigned)W, (unsigned)ceil_div(nqb, MASK_QT));
        SD_TRY(prof_begin(ctx, SD_PHASE_BD_MASKS));
        bd_mask_kernel<<<mgrid, 128, 0, st>>>(dX, T, n, ld, d_q + q0, nqb, (int)W, M, ctx->d_status);
        SD_TRY(prof_end(ctx));
        ctx->last.launches++;
        SD_TRY(prof_begin(ctx, SD_PHASE_BD_PAIRS));
        if (j == 2) {
            dim3 pgrid((unsigned)ceil_div(m, PAIR_TJ), (unsigned)nqb);
            bd_pair_kernel<<<pgrid, PAIR_THREADS, 0, st>>>(M, m, (int)W, d_out + q0, d_hits);
        } else {
            const i64 npairs = m * (m - 1) / 2;
            dim3 tgrid((unsigned)ceil_div(npairs, 256), (unsigned)nqb);
            bd_triple_kernel<<<tgrid, 256, 0, st>>>(M, m, (int)W, d_out + q0);
        }
        SD_TRY(prof_end(ctx));
        ctx->last.launches++;
        SD_CUDA(cudaGetLastError());
    }
    return SD_OK;
}

}  // namespace sd
