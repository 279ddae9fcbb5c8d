// modal.cu -- h-modal depth (K15): a curve is the vector of its F = T d values and
//   S_q = sum_j exp(c d2(x_q, x_j)),   c = -1 / (2 h^2),   depth = S_q phi(0) / n_pop (formed by the host),
// with the bandwidth h a quantile of the n (n - 1) / 2 pair distances (the host interpolates two order statistics).
//
// Both passes recompute d2 with pairdist.cuh's FP64 tile (query tile x sample tile blocks, f in order):
//   sum pass     one partial per (query, sample tile): exp(c d2) summed over the tile's columns in a fixed order (each
//                thread walks its 8 columns in order, then a fixed butterfly over the 16 lanes of a row); the finish
//                kernel adds a query's partials in tile order.  The grid spans the sample tiles, so one query against
//                100 000 curves runs 782 blocks.  No float atomics: a query's S depends on nothing but the two rows
//                of each pair and the tile sizes.  Out of sample the query's own row is column nS (d2 = 0, exp(-0) =
//                1), where the in-sample call of the sample with the query appended has it.
//   selection    the k-th and k1-th smallest d2 over the pairs i < j: the u64 bit patterns of d2 >= 0 sort like
//                the values, so a radix select over their digits finds them exactly.  Histogram passes over the
//                pair tiles (exact integer counts: per-block u32 sub-histograms, warp-aggregated, merged into u64)
//                narrow each target to a bin; once the bins hold at most MD_CAND_BUDGET bytes of keys one more pass
//                gathers them, and the remaining digits are resolved on that buffer at memory speed.  Bins too large
//                to gather are resolved by further pair passes down to the last digit.  The pair set is never
//                materialised.
#include <float.h>

#include <algorithm>
#include <cstring>
#include <vector>

#include "pairdist.cuh"

namespace sd {

constexpr size_t MD_PART_BUDGET = 256ull << 20;  // bytes of one row block of sum-pass partials (BUF_MODAL)
constexpr size_t MD_CAND_BUDGET = 1ull << 30;    // bytes of gathered candidate keys (BUF_MODAL)
constexpr int MD_BINS = 4096;                    // 12-bit digits
constexpr int MD_NPASS = 6;
constexpr int MD_SHIFT[MD_NPASS] = {52, 40, 28, 16, 4, 0};
constexpr int MD_WIDTH[MD_NPASS] = {12, 12, 12, 12, 12, 4};

// grid (ceil(ncol / SP_BS), ceil(nq / SP_BQ)), ncol = nS + (self_col >= 0).  part[q * gridDim.x + blockIdx.x] = the
// sum over this tile's columns s < ncol of exp(c d2(Q[idx(q)], S[s])), d2 taken as 0 at s == self_col.
__global__ void __launch_bounds__(SP_THREADS) modal_sum_kernel(const double *__restrict__ Q,
                                                               const i64 *__restrict__ qidx, const i64 nq,
                                                               const double *__restrict__ S, const i64 nS,
                                                               const i64 self_col, const i64 F, const double c,
                                                               double *__restrict__ part, int *__restrict__ status) {
    __shared__ __align__(16) double As[2][SP_BK][SP_BQ];
    __shared__ __align__(16) double Bs[2][SP_BK][SP_BS];
    const int tx = threadIdx.x % 16, ty = threadIdx.x / 16;
    const i64 q0 = (i64)blockIdx.y * SP_BQ, s0 = (i64)blockIdx.x * SP_BS;
    const i64 ncol = self_col >= 0 ? nS + 1 : nS;
    double acc[SP_TQ][SP_TS];
#pragma unroll
    for (int i = 0; i < SP_TQ; ++i)
#pragma unroll
        for (int j = 0; j < SP_TS; ++j) acc[i][j] = 0.0;
    sq_dist_tile(As, Bs, tx, ty, Q, qidx, q0, nq, S, s0, nS, F, acc);
    bool overflow = false;
#pragma unroll
    for (int i = 0; i < SP_TQ; ++i) {
        const i64 q = q0 + ty + 16 * i;
        double v = 0.0;
#pragma unroll
        for (int j = 0; j < SP_TS; ++j) {
            const i64 s = s0 + tx + 16 * j;
            const double d2 = s == self_col ? 0.0 : acc[i][j];
            if (q < nq && s < ncol) {
                if (!(d2 <= DBL_MAX)) overflow = true;
                v = __dadd_rn(v, exp(__dmul_rn(c, d2)));
            }
        }
        // the 16 lanes of one ty: a fixed butterfly, every lane ends with the same bits
#pragma unroll
        for (int m = 1; m < 16; m <<= 1) v = __dadd_rn(v, __shfl_xor_sync(0xffffffffu, v, m));
        if (tx == 0 && q < nq) part[q * gridDim.x + blockIdx.x] = v;
    }
    if (overflow) atomicOr(status, ST_OVERFLOW);
}

__global__ void modal_finish_kernel(const double *__restrict__ part, const i64 nq, const i64 ntile,
                                    double *__restrict__ out) {
    const i64 q = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= nq) return;
    double v = 0.0;
    for (i64 t = 0; t < ntile; ++t) v = __dadd_rn(v, part[q * ntile + t]);
    out[q] = v;
}

// Which of the (at most two) targets a key counts for: the bin (digit) in h[0 .. MD_BINS) when (key & mask) == pa,
// else in h[MD_BINS ..) when two and (key & mask) == pb; -1 for neither.
struct SelPass {
    u64 mask, pa, pb;
    int shift, width, two;
    __device__ __forceinline__ int bin(const u64 key) const {
        const int digit = (int)((key >> shift) & ((1ull << width) - 1));
        if ((key & mask) == pa) return digit;
        if (two && (key & mask) == pb) return MD_BINS + digit;
        return -1;
    }
};

// one warp-aggregated shared-memory increment per distinct bin of the warp's 32 lanes (all lanes call it)
__device__ __forceinline__ void hist_add(unsigned *h, const int bin) {
    const unsigned peers = __match_any_sync(0xffffffffu, bin);
    if (bin >= 0 && (threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(&h[bin], (unsigned)__popc(peers));
}

// one warp-aggregated append of the keys of the lanes with take set (all lanes call it)
__device__ __forceinline__ void gather_add(u64 *cand, unsigned long long *ncand, const u64 cap, const bool take,
                                           const u64 key) {
    const unsigned ballot = __ballot_sync(0xffffffffu, take);
    if (!ballot) return;
    const int lane = threadIdx.x & 31, leader = __ffs(ballot) - 1;
    unsigned long long base = 0;
    if (lane == leader) base = atomicAdd(ncand, (unsigned long long)__popc(ballot));
    base = __shfl_sync(0xffffffffu, base, leader);
    const u64 at = base + __popc(ballot & ((1u << lane) - 1));
    if (take && at < cap) cand[at] = key;
}

__device__ __forceinline__ void hist_flush(unsigned *h, const int nbins, unsigned long long *ghist) {
    __syncthreads();
    for (int e = threadIdx.x; e < nbins; e += SP_THREADS)
        if (h[e]) atomicAdd(&ghist[e], (unsigned long long)h[e]);
}

// grid (ceil(n / SP_BS), ceil(n / SP_BQ)) over the pairs i < j of the rows X [n, F]: GATHER appends the keys the pass
// selects (mask 0 selects all) to cand, else their digits are counted into ghist [2][MD_BINS].  Blocks holding no
// pair i < j exit at once; a d2 that overflows sets ST_OVERFLOW (its key, +inf, still sorts last).
template <bool GATHER>
__global__ void __launch_bounds__(SP_THREADS) modal_pairs_kernel(const double *__restrict__ X, const i64 n,
                                                                 const i64 F, const SelPass p,
                                                                 unsigned long long *__restrict__ ghist,
                                                                 u64 *__restrict__ cand,
                                                                 unsigned long long *__restrict__ ncand,
                                                                 const u64 cap, int *__restrict__ status) {
    __shared__ __align__(16) double tile[2 * SP_BK * (SP_BQ + SP_BS)];  // As, Bs; then the sub-histograms
    double (*As)[SP_BK][SP_BQ] = reinterpret_cast<double (*)[SP_BK][SP_BQ]>(tile);
    double (*Bs)[SP_BK][SP_BS] = reinterpret_cast<double (*)[SP_BK][SP_BS]>(tile + 2 * SP_BK * SP_BQ);
    const int tx = threadIdx.x % 16, ty = threadIdx.x / 16;
    const i64 q0 = (i64)blockIdx.y * SP_BQ, s0 = (i64)blockIdx.x * SP_BS;
    if (s0 + SP_BS - 1 <= q0) return;  // every j <= every i
    double acc[SP_TQ][SP_TS];
#pragma unroll
    for (int i = 0; i < SP_TQ; ++i)
#pragma unroll
        for (int j = 0; j < SP_TS; ++j) acc[i][j] = 0.0;
    sq_dist_tile(As, Bs, tx, ty, X, nullptr, q0, n, X, s0, n, F, acc);
    unsigned *h = reinterpret_cast<unsigned *>(tile);  // 2 MD_BINS u32: 32 KB of the 48 KB
    const int nbins = p.two ? 2 * MD_BINS : MD_BINS;
    if (!GATHER) {
        for (int e = threadIdx.x; e < nbins; e += SP_THREADS) h[e] = 0;
        __syncthreads();
    }
    bool overflow = false;
#pragma unroll
    for (int i = 0; i < SP_TQ; ++i) {
        const i64 q = q0 + ty + 16 * i;
#pragma unroll
        for (int j = 0; j < SP_TS; ++j) {
            const i64 s = s0 + tx + 16 * j;
            const bool pair = q < n && s < n && s > q;
            const double d2 = acc[i][j];
            if (pair && !(d2 <= DBL_MAX)) overflow = true;
            const u64 key = (u64)__double_as_longlong(d2);
            const int bin = pair ? p.bin(key) : -1;
            if (GATHER) gather_add(cand, ncand, cap, bin >= 0, key);
            else hist_add(h, bin);
        }
    }
    if (!GATHER) hist_flush(h, nbins, ghist);
    if (overflow) atomicOr(status, ST_OVERFLOW);
}

// the same count over m gathered keys (grid-stride)
__global__ void __launch_bounds__(SP_THREADS) modal_cand_hist_kernel(const u64 *__restrict__ cand, const i64 m,
                                                                     const SelPass p,
                                                                     unsigned long long *__restrict__ ghist) {
    __shared__ unsigned h[2 * MD_BINS];
    const int nbins = p.two ? 2 * MD_BINS : MD_BINS;
    for (int e = threadIdx.x; e < nbins; e += SP_THREADS) h[e] = 0;
    __syncthreads();
    const i64 stride = (i64)gridDim.x * SP_THREADS;
    const i64 end = ceil_div(m, stride) * stride;  // whole warps run every iteration
    for (i64 e = (i64)blockIdx.x * SP_THREADS + threadIdx.x; e < end; e += stride)
        hist_add(h, e < m ? p.bin(cand[e]) : -1);
    hist_flush(h, nbins, ghist);
}

namespace {

struct Target {
    u64 prefix = 0;
    i64 rank = 0;  // within the keys that share prefix on the digits resolved so far
    i64 count = 0;  // how many keys share it
};

// the bin of h [MD_BINS] holding t.rank; narrows t to it
void narrow(Target &t, const u64 *h, const int shift) {
    i64 below = 0;
    for (int b = 0; b < MD_BINS; ++b) {
        const i64 c = (i64)h[b];
        if (t.rank < below + c) {
            t.prefix |= (u64)b << shift;
            t.rank -= below;
            t.count = c;
            return;
        }
        below += c;
    }
    t.count = 0;  // unreachable while the counts are exact
}

}  // namespace

// the k0-th and k1-th smallest (0-based) squared distances over the pairs i < j of the rows dX [n, F]
int modal_select_device(sd_ctx *ctx, const double *dX, i64 n, i64 F, i64 k0, i64 k1, double *out) {
    const i64 npairs = n * (n - 1) / 2;
    cudaStream_t st = ctx->stream;
    SD_TRY(ctx->buf[BUF_AUX].reserve((2 * MD_BINS + 1) * sizeof(unsigned long long)));
    unsigned long long *ghist = ctx->buf[BUF_AUX].as<unsigned long long>();
    unsigned long long *ncand = ghist + 2 * MD_BINS;
    const i64 cap = (i64)(MD_CAND_BUDGET / sizeof(u64));
    const dim3 pgrid((unsigned)ceil_div(n, SP_BS), (unsigned)ceil_div(n, SP_BQ));
    std::vector<u64> h(2 * MD_BINS);
    Target t[2];
    t[0].rank = k0;
    t[1].rank = k1;
    t[0].count = t[1].count = npairs;
    u64 mask = 0;
    u64 *cand = nullptr;
    i64 m = 0;  // gathered keys
    auto gather = [&](const SelPass &p, i64 total) -> int {
        SD_TRY(ctx->buf[BUF_MODAL].reserve((size_t)total * sizeof(u64)));
        cand = ctx->buf[BUF_MODAL].as<u64>();
        SD_CUDA(cudaMemsetAsync(ncand, 0, sizeof(unsigned long long), st));
        modal_pairs_kernel<true><<<pgrid, SP_THREADS, 0, st>>>(dX, n, F, p, ghist, cand, ncand, (u64)total,
                                                               ctx->d_status);
        ctx->last.launches += 1;
        SD_CUDA(cudaGetLastError());
        m = total;
        return SD_OK;
    };
    if (npairs <= cap) SD_TRY(gather(SelPass{0, 0, 0, 0, 0, 0}, npairs));
    for (int pass = 0; pass < MD_NPASS; ++pass) {
        const SelPass p{mask, t[0].prefix, t[1].prefix, MD_SHIFT[pass], MD_WIDTH[pass], t[0].prefix != t[1].prefix};
        SD_CUDA(cudaMemsetAsync(ghist, 0, 2 * MD_BINS * sizeof(unsigned long long), st));
        if (cand) {
            const int blocks = (int)std::min<i64>(ceil_div(m, SP_THREADS * 8), 4ll * ctx->sm_count);
            modal_cand_hist_kernel<<<blocks > 0 ? blocks : 1, SP_THREADS, 0, st>>>(cand, m, p, ghist);
        } else {
            modal_pairs_kernel<false><<<pgrid, SP_THREADS, 0, st>>>(dX, n, F, p, ghist, nullptr, nullptr, 0,
                                                                    ctx->d_status);
        }
        ctx->last.launches += 1;
        SD_CUDA(cudaGetLastError());
        SD_CUDA(cudaMemcpyAsync(h.data(), ghist, 2 * MD_BINS * sizeof(u64), cudaMemcpyDeviceToHost, st));
        SD_CUDA(cudaStreamSynchronize(st));
        const bool two = p.two;
        narrow(t[0], h.data(), p.shift);
        narrow(t[1], h.data() + (two ? MD_BINS : 0), p.shift);
        if (t[0].count == 0 || t[1].count == 0) {
            set_error("modal pair selection: lost the target rank (internal error)");
            return SD_ERR_INVALID;
        }
        mask |= ((1ull << p.width) - 1) << p.shift;
        if (!cand && pass + 1 < MD_NPASS) {
            const bool split = t[0].prefix != t[1].prefix;
            const i64 total = t[0].count + (split ? t[1].count : 0);
            if (total <= cap) SD_TRY(gather(SelPass{mask, t[0].prefix, t[1].prefix, 0, 0, split}, total));
        }
    }
    for (int i = 0; i < 2; ++i) memcpy(&out[i], &t[i].prefix, sizeof(double));
    return SD_OK;
}

// S_q of the nq queries (rows dQ[idx(q) * F], idx = d_qidx or q) against the sample rows dS [nS, F]; with self set,
// each query is also column nS of its own row (out of sample).  Row blocks of queries keep the partials within
// MD_PART_BUDGET; a query's bits do not depend on the row block.
int modal_sums_device(sd_ctx *ctx, const double *dQ, const i64 *d_qidx, i64 nq, const double *dS, i64 nS, i64 F,
                      bool self, double c, double *d_out) {
    if (nq == 0) return SD_OK;
    const i64 ncol = nS + (self ? 1 : 0);
    const i64 ntile = ceil_div(ncol, SP_BS);
    i64 RB = (i64)(MD_PART_BUDGET / ((size_t)ntile * sizeof(double))) / SP_BQ * SP_BQ;
    if (RB < SP_BQ) RB = SP_BQ;
    if (RB > 65535ll * SP_BQ) RB = 65535ll * SP_BQ;  // grid.y
    if (RB > ceil_div(nq, SP_BQ) * SP_BQ) RB = ceil_div(nq, SP_BQ) * SP_BQ;
    SD_TRY(ctx->buf[BUF_MODAL].reserve((size_t)RB * ntile * sizeof(double)));
    double *dPart = ctx->buf[BUF_MODAL].as<double>();
    cudaStream_t st = ctx->stream;
    for (i64 r0 = 0; r0 < nq; r0 += RB) {
        const i64 rows = nq - r0 < RB ? nq - r0 : RB;
        const double *Q = d_qidx ? dQ : dQ + r0 * F;
        const i64 *qi = d_qidx ? d_qidx + r0 : nullptr;
        modal_sum_kernel<<<dim3((unsigned)ntile, (unsigned)ceil_div(rows, SP_BQ)), SP_THREADS, 0, st>>>(
            Q, qi, rows, dS, nS, self ? nS : -1, F, c, dPart, ctx->d_status);
        modal_finish_kernel<<<(unsigned)ceil_div(rows, 256), 256, 0, st>>>(dPart, rows, ntile, d_out + r0);
        ctx->last.launches += 2;
        SD_CUDA(cudaGetLastError());
    }
    return SD_OK;
}

}  // namespace sd
