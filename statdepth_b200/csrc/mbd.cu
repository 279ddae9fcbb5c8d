// mbd.cu -- modified band depth (relax=True): per-time-row strict ranks on sm_100a.
//
// Replaces the relaxed branch of _r2_containment (statdepth/depth/calculations/_containment.py:68-80)
// summed over all j-subsets by _univariate_band_depth (_functional.py:238-253).  For one time row,
// with b / a = number of OTHER curves strictly below / above curve c,
//     #{j-subsets whose closed band contains c} = C(n-1,j) - C(b,j) - C(a,j)
// so the whole relaxed numerator is a per-row ranking problem (SURVEY 8a row a3, kernel "K1").
//
// Two pipelines produce the same integers.  Rows of 16 384 .. 131 072 curves take the SLAB path of mbd_slab.cuh
// (included below: the row stays on the chip, three CTAs per row sort whole bins per thread); this file holds the
// PART pipeline, which ranks every other row length, the rows the slab path declines (ties, wild tails; under a row
// mask) and everything under SD_MBD_PATH=parts, and the driver that chooses (rank_pipeline).  It has two fronts:
// mbd_all_device accumulates the relaxed numerators, rank_rows_device writes the ranks b and a of every value.
//
// Part pipeline per block of time rows (all kernels on ctx->stream, no host sync):
//   1. mbd_splitters_kernel : one CTA per row sorts a strided sample (u32 images of float(x - ref), register
//                             bitonic network per warp + swizzled shared-memory merges) and emits P-1
//                             equal-mass splitters.
//   2. mbd_partition_kernel : streams the row once from HBM, finds each value's part with a bucket table,
//                             groups a 4096-value chunk by part in shared memory (one shared atomic per
//                             value, one global atomic per (CTA, part)) and copies the groups to the parts'
//                             slot lists (fixed capacity CAP) with coalesced stores.  Equal values always
//                             share a part, so tie runs never straddle parts.  A list entry is 8 bytes: the
//                             value as a FLOAT offset from the part's lower splitter (monotone in x, resolution
//                             2^-24 of the part's width) and the curve id.
//   3. mbd_rank_kernel      : ONE WARP per (row, part): loads <= 512 offsets, maps them to a 22-bit
//                             monotone key packed with the slot id, sorts the packed u32 keys in
//                             registers with a shuffle bitonic network, resolves equal-key runs with
//                             exact fp64 compares on the values of X (gathered through the curve ids; rare),
//                             and adds b(b-1) + a(a-1) to raw[curve] with a 64-bit RED.
//      mbd_rank_big_kernel  : persistent; drains the work list of parts with 513..1024 values.
//      mbd_heavy_kernel     : one CTA per row, before the rank kernels: writes the exclusive prefix of the part
//                             sizes (#values in lower parts) for them; rows with parts of more than CAP values
//                             (a few heavily repeated values: ties) rank those parts from a per-part table of
//                             at most 8 distinct values, no sorting.
//   4. mbd_fallback_kernel  : rows in which a part of more than CAP values holds more than 8 distinct values
//                             (adversarial spreads) are ranked by a generic one-CTA-per-row bitonic
//                             sort of order-preserving u64 keys + binary-search ranks (persistent over the rows:
//                             almost always none is flagged).  Correct for any finite input; slower.
//   5. mbd_finish_kernel    : numerator += rows * C(n-1,2) - raw / 2, once per call.
// Row groups (mbd_all_device(..., group_rows)): the rows may be G stacked matrices of equal shape that accumulate
// into [G][n] (batched permutations); rank_rows_device (no accumulator) skips the REDs.
// HBM layout: X[t*ld + c] float64 (time-major rows are contiguous and streamed with coalesced
// loads); raw uint64[n] -> acc int64[n] (mbd_finish_kernel); part lists [row][part][CAP] float32 + uint32.
#include <stdlib.h>

#include "common.cuh"
#include "sortnet.cuh"

namespace sd {

constexpr int CAP = 1024;          // slots per part == max elements one warp ranks
constexpr int TARGET_PART = 400;   // mean part size the splitter count aims for
constexpr int MAX_PARTS = 1024;
constexpr int MAX_SAMPLE = 8192;   // 64 KB of shared memory in the splitter kernel
constexpr int OVERSAMPLE = 32;     // sample elements per part
constexpr int KEY_BITS = 22;       // reduced key bits (10 low bits carry the slot id)
constexpr u32 KEY_MAX = (1u << KEY_BITS) - 1u;
constexpr int FB_TILE = 4096;      // keys sorted in shared memory by the fallback
constexpr int PT_BUCKETS = 1024;   // partition: equal-width lookup table over the splitter range

__device__ __forceinline__ i64 comb2_dev(i64 m) { return m * (m - 1) / 2; }
__device__ __forceinline__ i64 comb3_dev(i64 m) {
    // m(m-1)/2 is exact; (m(m-1)/2)*(m-2) is divisible by 3; fits in int64 for m < 2.6e6
    return m < 3 ? 0 : (m * (m - 1) / 2) * (m - 2) / 3;
}

// ---------------------------------------------------------------------------------------------
// 1. splitters: one CTA per row sorts a strided sample of S = 1024*W values (W = 1, 2, 4 or 8 warps)
//    as order-preserving u32 images of float(x - ref) -- splitters need not be data values, any
//    non-decreasing sequence works, and 32-bit keys sort on registers at 2 instructions per
//    compare-exchange.  Each warp sorts 1024 keys (EPL = 32); the 1..3 remaining merge levels exchange
//    partners through XOR-swizzled shared memory and finish on registers.  v1 (fp64 bitonic in shared
//    memory, 91 block-wide stages) took 0.56 ms of a 3.6 ms step.
// ---------------------------------------------------------------------------------------------
constexpr int SP_THREADS = 256;

// Reference value of a row: splitters and part lists work on float(x - reference), so the reference has to
// sit inside the bulk of the row or the float offsets lose the differences between values.  The median of
// three entries survives one outlier; every kernel recomputes it the same way.
__device__ __forceinline__ double row_reference(const double *__restrict__ xr, const i64 n) {
    const double a = xr[0], b = xr[n >> 1], c = xr[n - 1];
    return fmax(fmin(a, b), fmin(fmax(a, b), c));
}

__device__ __forceinline__ u32 f32_sortable(float f) {
    const u32 b = __float_as_uint(f);
    return b ^ ((b & 0x80000000u) ? 0xffffffffu : 0x80000000u);
}
__device__ __forceinline__ float f32_unsortable(u32 k) {
    return __uint_as_float(k ^ ((k & 0x80000000u) ? 0x80000000u : 0xffffffffu));
}
__device__ __forceinline__ int sp_swz(int g) { return g ^ ((g >> 5) & 31); }

__global__ void __launch_bounds__(SP_THREADS) mbd_splitters_kernel(const double *__restrict__ X, i64 n, i64 ld,
                                                                   int P, int S, float *__restrict__ splitters_f,
                                                                   unsigned short *__restrict__ tables,
                                                                   int *__restrict__ rowflag, int *__restrict__ status,
                                                                   const int *__restrict__ only) {
    if (only && !(only[blockIdx.x] & 2)) return;  // masked call: only the rows the slab path gave up
    __shared__ u32 skey[MAX_SAMPLE];
    __shared__ float s_splf[MAX_PARTS];
    __shared__ int s_dups;
    if (threadIdx.x == 0) s_dups = 0;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int W = S >> 10;  // warps that hold samples
    const double *xr = X + (i64)blockIdx.x * ld;
    const double x0 = row_reference(xr, n);
    u32 v[32];
    if (wid < W) {
        bool bad = false;
        // strided sample taken in quads of 4 consecutive values (one 32 B sector each)
        const i64 nquad = n >> 2;
        const int squad_shift = __ffs(S >> 2) - 1;  // S is a power of two
#pragma unroll
        for (int i = 0; i < 32; ++i) {
            const int g = wid * 1024 + lane * 32 + i;
            const i64 idx = (((i64)(g >> 2) * nquad) >> squad_shift) * 4 + (g & 3);
            const double x = xr[idx];
            bad |= !isfinite(x);
            v[i] = f32_sortable(__double2float_rn(x - x0));
        }
        if (bad) atomicOr(status, ST_NONFINITE);
        warp_bitonic_sort<32, u32>(v, lane);
    }
    for (int k = 2048; k <= S; k <<= 1) {  // merge levels wider than one warp
        for (int j = k; j >= 2048; j >>= 1) {  // j == k: mirror stage (g ^ (k-1)); else xor stage (g ^ j/2)
            __syncthreads();
            if (wid < W) {
#pragma unroll
                for (int i = 0; i < 32; ++i) skey[sp_swz(wid * 1024 + lane * 32 + i)] = v[i];
            }
            __syncthreads();
            if (wid < W) {
                const int xorv = (j == k) ? (k - 1) : (j >> 1);
                const bool lower = ((wid * 1024) & (j == k ? (k >> 1) : (j >> 1))) == 0;
#pragma unroll
                for (int i = 0; i < 32; ++i) {
                    const u32 o = skey[sp_swz((wid * 1024 + lane * 32 + i) ^ xorv)];
                    v[i] = lower ? min(v[i], o) : max(v[i], o);
                }
            }
        }
        if (wid < W) warp_merge_tail<32, u32>(v, lane, 16);  // strides 512 .. 1 stay inside the warp
    }
    __syncthreads();
    if (wid < W) {
        // tie-heavy rows (rounded data: every part holds a handful of values): a quarter of the sorted sample repeating
        // its neighbour means the sub-bin ranking cannot work (all copies of a value share a bin) -- bit 2 of the row's
        // flag sends its parts straight to the sorting network
        int dups = 0;
#pragma unroll
        for (int i = 0; i + 1 < 32; ++i) dups += v[i] == v[i + 1];
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) dups += __shfl_xor_sync(0xffffffffu, dups, d);
        if (lane == 0) atomicAdd(&s_dups, dups);
#pragma unroll
        for (int i = 0; i < 32; ++i) skey[sp_swz(wid * 1024 + lane * 32 + i)] = v[i];
    }
    __syncthreads();
    if (threadIdx.x == 0 && 4 * s_dups > S) atomicOr(&rowflag[blockIdx.x], 4);
    // splitter p as a float offset from the row reference: what the partition compares, and the reference the part
    // lists store their values against
    float *outf = splitters_f + (i64)blockIdx.x * (P - 1);
    const int nspl = P - 1;
    for (int p = tid + 1; p < P; p += SP_THREADS) s_splf[p - 1] = f32_unsortable(skey[sp_swz((int)(((i64)p * S) / P))]);
    __syncthreads();
    // A value repeated so often that it takes several splitter positions (v v v w) gets a part of its own:
    // the repeats become the next float up (v v+ v+ w), so that [v, v+) holds exactly the values whose
    // offset rounds to v and the values above v are not lumped with them into one over-full part.
    float mine[(MAX_PARTS + SP_THREADS - 1) / SP_THREADS];
#pragma unroll
    for (int k = 0; k < (MAX_PARTS + SP_THREADS - 1) / SP_THREADS; ++k) {
        const int i = tid + k * SP_THREADS;
        float f = 0.f;
        if (i < nspl) {
            f = s_splf[i];
            if (i > 0 && s_splf[i - 1] == f) f = nextafterf(f, INFINITY);
        }
        mine[k] = f;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < (MAX_PARTS + SP_THREADS - 1) / SP_THREADS; ++k) {
        const int i = tid + k * SP_THREADS;
        if (i < nspl) {
            s_splf[i] = mine[k];
            outf[i] = mine[k];
        }
    }
    __syncthreads();
    // lookup table for the partition kernel: tbl[b] = #splitters < lower edge of equal-width bucket b over
    // [first splitter, last splitter]; built once per row here instead of once per partition CTA
    const float f_first = s_splf[0];
    const float w = (s_splf[nspl - 1] - f_first) * (1.0f / PT_BUCKETS);
    const bool usable = w > 0.f && w < INFINITY;
    int top = 1;
    while (top < P) top <<= 1;
    unsigned short *tbl = tables + (i64)blockIdx.x * PT_BUCKETS;
    for (int b = tid; b < PT_BUCKETS; b += SP_THREADS) {
        const float edge = f_first + (float)b * w;
        int lo = 0;
        for (int step = top >> 1; step > 0; step >>= 1) {
            const int probe = lo + step;
            if (probe <= nspl && s_splf[probe - 1] < edge) lo = probe;
        }
        tbl[b] = (unsigned short)(usable ? lo : 0);
    }
}

// ---------------------------------------------------------------------------------------------
// 2. partition: one CTA groups a chunk of PT_CHUNK values of one row by part in shared memory
//    (shared-memory atomics give the position inside the CTA's group), reserves a contiguous slot
//    range per part with ONE global atomic per (CTA, part), and copies the groups out with
//    coalesced stores.  (v1 did one global atomic + two scattered 8/4-byte stores per value and
//    was bound by L2 atomic / sector-write throughput: 2.1 ms of a 4.2 ms step.)
// ---------------------------------------------------------------------------------------------
#ifndef SD_PT_THREADS
#define SD_PT_THREADS 256
#endif
#ifndef SD_PT_EPT
#define SD_PT_EPT 16
#endif
#ifndef SD_PT_MINB
#define SD_PT_MINB (SD_PT_THREADS >= 512 ? 2 : 3)  // resident CTAs per SM the register budget is held to
#endif
constexpr int PT_THREADS = SD_PT_THREADS;
constexpr int PT_EPT = SD_PT_EPT;               // values per thread
constexpr int PT_CHUNK = PT_THREADS * PT_EPT;   // 4096 values per CTA
constexpr size_t PT_SMEM = (size_t)PT_CHUNK * 4 + (size_t)PT_CHUNK * 4 + (size_t)(MAX_PARTS * 3 + 4) * 4 +
                           (size_t)(PT_BUCKETS + 8) * 2 + 256;

// part of a value = number of splitters <= f, f = float(x - ref).  Every step is monotone in x, so
// equal values share a part and parts are ordered.  sp[] is the row's splitter list padded with sentinels:
// sp[0] = NaN, sp[1 + i] = splitter i, sp[nspl + 1] = sp[nspl + 2] = NaN (every compare with a sentinel is
// false, also for f = +-inf, so the scans stop at the ends).  The lookup table only provides
// a starting guess (first splitter of the value's equal-width bucket); three independent shared loads around
// the guess settle almost every value, the two scans behind them make the result exact for all.
constexpr int SPL_PAD = 3;
__device__ __forceinline__ void fill_splitters(float *sp, const float *__restrict__ row_splitters, const int nspl,
                                               const int tid, const int nthreads) {
    for (int i = tid; i < nspl; i += nthreads) sp[1 + i] = row_splitters[i];
    if (tid == 0) {
        sp[0] = NAN;
        sp[nspl + 1] = NAN;
        sp[nspl + 2] = NAN;
    }
}

// `lower` receives sp[part], the splitter below the part (NaN for part 0).
__device__ __forceinline__ int part_of(const float f, const float *__restrict__ sp, const unsigned short *__restrict__ tbl,
                                       const float f_first, const float inv_w, float &lower) {
    float fb = (f - f_first) * inv_w;
    fb = fminf(fmaxf(fb, 0.f), (float)(PT_BUCKETS - 1));  // also maps NaN (inf * 0) to 0
    int idx = tbl[(int)fb];
    const float below = sp[idx], s0 = sp[idx + 1], s1 = sp[idx + 2];
    if (below > f) {  // guess too high (bucket rounding): rare
        do --idx; while (sp[idx] > f);
        lower = sp[idx];
        return idx;
    }
    const bool ge0 = s0 <= f, ge1 = s1 <= f;
    idx += (int)ge0 + (int)ge1;
    lower = ge1 ? s1 : (ge0 ? s0 : below);
    if (ge1) {  // more than two splitters of this bucket are <= f: rare
        while (sp[idx + 1] <= f) ++idx;
        lower = sp[idx];
    }
    return idx;
}

__global__ void __launch_bounds__(PT_THREADS, SD_PT_MINB) mbd_partition_kernel(const double *__restrict__ X, i64 n, i64 ld, int P,
                                                                   const float *__restrict__ splitters_f,
                                                                   const unsigned short *__restrict__ tables,
                                                                   int *__restrict__ cursor, int *__restrict__ rowflag,
                                                                   float *__restrict__ part_x,
                                                                   u32 *__restrict__ part_j, i64 row_stride,
                                                                   int *__restrict__ status,
                                                                   const int *__restrict__ only) {
    if (only && !(only[blockIdx.y] & 2)) return;
    extern __shared__ __align__(16) unsigned char pt_smem[];
    float *sx = reinterpret_cast<float *>(pt_smem);                   // grouped values (offsets from the part's reference)
    u32 *sj = reinterpret_cast<u32 *>(sx + PT_CHUNK);                 // grouped (part << 12 | index in chunk)
    float *splf = reinterpret_cast<float *>(sj + PT_CHUNK);           // splitters of this row (float offsets)
    int *pre = reinterpret_cast<int *>(splf + MAX_PARTS + 4);         // per-part count, then exclusive prefix
    int *off = pre + MAX_PARTS;                                       // global slot base - prefix
    unsigned short *tbl = reinterpret_cast<unsigned short *>(off + MAX_PARTS);  // bucket -> first splitter
    int *wtot = reinterpret_cast<int *>(tbl + PT_BUCKETS + 8);        // warp totals of the scan

    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int row = blockIdx.y;
    const double *xr = X + (i64)row * ld;
    const int nspl = P - 1;
    const i64 c0 = (i64)blockIdx.x * PT_CHUNK;
    const int len = (n - c0) < PT_CHUNK ? (int)(n - c0) : PT_CHUNK;

    // A. load (issued before the row's tables are staged, so both latencies overlap), locate the part, claim a
    //    position inside the CTA's group (shared-memory atomic)
    double x[PT_EPT];
    u32 tag[PT_EPT];  // part << 16 | position within (CTA, part)
    float rel[PT_EPT];  // value as a float offset from the part's lower splitter (part 0: from the first splitter)
#pragma unroll
    for (int u = 0; u < PT_EPT; ++u) {
        const int i = u * PT_THREADS + tid;
        x[u] = i < len ? xr[c0 + i] : 0.0;
    }
    const double x0 = row_reference(xr, n);
    fill_splitters(splf, splitters_f + (i64)row * nspl, nspl, tid, PT_THREADS);
    for (int i = tid; i < P; i += PT_THREADS) pre[i] = 0;
    for (int b = tid; b < PT_BUCKETS; b += PT_THREADS) tbl[b] = nspl > 0 ? tables[(i64)row * PT_BUCKETS + b] : 0;
    __syncthreads();
    float f_first = 0.f, inv_w = 0.f;
    if (nspl > 0) {
        f_first = splf[1];
        const float w = (splf[nspl] - f_first) * (1.0f / PT_BUCKETS);
        if (w > 0.f && w < INFINITY) inv_w = 1.0f / w;
    }
    bool bad = false;
#pragma unroll
    for (int u = 0; u < PT_EPT; ++u) bad |= !isfinite(x[u]);
#pragma unroll
    for (int u = 0; u < PT_EPT; ++u) {
        const int i = u * PT_THREADS + tid;
        tag[u] = 0xffffffffu;
        rel[u] = 0.f;
        if (i < len) {
            const double d = x[u] - x0;
            int part = 0;
            double ref = 0.0;
            if (nspl > 0) {
                float lower;
                part = part_of(__double2float_rn(d), splf, tbl, f_first, inv_w, lower);
                ref = (double)(part > 0 ? lower : f_first);
            }
            rel[u] = __double2float_rn(d - ref);  // monotone in x; 2^-24 of the part's width, not of |x - x0|
            tag[u] = ((u32)part << 16) | (u32)atomicAdd(&pre[part], 1);
        }
    }
    if (bad) atomicOr(status, ST_NONFINITE);
    __syncthreads();

    // B. exclusive scan of the per-part counts; one global atomic per non-empty part reserves its slots
    {
        const int ppt = (P + PT_THREADS - 1) / PT_THREADS;  // <= 4
        const int p0 = tid * ppt;
        int cnt[4] = {0, 0, 0, 0}, run = 0;
#pragma unroll
        for (int k = 0; k < 4; ++k)
            if (k < ppt && p0 + k < P) { cnt[k] = pre[p0 + k]; run += cnt[k]; }
        int incl = run;
#pragma unroll
        for (int s = 1; s < 32; s <<= 1) {
            const int v = __shfl_up_sync(0xffffffffu, incl, s);
            if (lane >= s) incl += v;
        }
        if (lane == 31) wtot[wid] = incl;
        __syncthreads();
        int base = incl - run;
        for (int w = 0; w < wid; ++w) base += wtot[w];
        bool over = false;
        int *cur = cursor + (i64)row * P;
#pragma unroll
        for (int k = 0; k < 4; ++k)
            if (k < ppt && p0 + k < P) {
                int g = 0;
                if (cnt[k] > 0) {
                    g = atomicAdd(&cur[p0 + k], cnt[k]);
                    over |= g + cnt[k] > CAP;
                }
                pre[p0 + k] = base;
                off[p0 + k] = g - base;
                base += cnt[k];
            }
        if (over) atomicOr(&rowflag[row], 1);  // bit 0: some part holds more than CAP values
    }
    __syncthreads();

    // C. group in shared memory
#pragma unroll
    for (int u = 0; u < PT_EPT; ++u) {
        if (tag[u] != 0xffffffffu) {
            const int part = (int)(tag[u] >> 16);
            const int pos = pre[part] + (int)(tag[u] & 0xffffu);
            sx[pos] = rel[u];
            sj[pos] = ((u32)part << 12) | (u32)(u * PT_THREADS + tid);
        }
    }
    __syncthreads();

    // D. coalesced copy-out: consecutive grouped positions of one part go to consecutive slots
    float *px = part_x + (i64)row * row_stride;
    u32 *pj = part_j + (i64)row * row_stride;
    for (int i = tid; i < len; i += PT_THREADS) {
        const u32 t = sj[i];
        const int part = (int)(t >> 12);
        const int slot = off[part] + i;
        if (slot < CAP) {
            const i64 at = (i64)part * CAP + slot;
            px[at] = sx[i];
            pj[at] = (u32)(c0 + (t & 4095u));
        }
    }
}

// ---------------------------------------------------------------------------------------------
// 3. per-part warp ranking
// ---------------------------------------------------------------------------------------------
struct RankOut {
    u64 *raw2;             // [n] sum over rows of b(b-1) + a(a-1); mbd_finish_kernel turns it into the j = 2 numerator
    i64 *acc3;             // j = 3 numerator, may be null
    int *rank_b, *rank_a;  // may be null (rank_a also when rank_b is given); [row_global*n + c]
    i64 n;
    i64 full2, full3;      // C(n-1,2), C(n-1,3)
    i64 group_rows;        // 0: one accumulator row; g > 0: rows [k*g, (k+1)*g) accumulate into row k of [G][n]
};

__device__ __forceinline__ i64 acc_offset(const RankOut &o, const i64 row_global) {
    return o.group_rows ? (row_global / o.group_rows) * o.n : 0;
}

// One (row, curve) result.  The j = 2 term C(n-1,2) - C(b,2) - C(a,2) is accumulated as the raw sum
// b(b-1) + a(a-1) (two 32x32->64 multiply-adds and one RED; m = 0 gives 0 * (2^32-1) = 0) and finished once
// per call by mbd_finish_kernel: numerator += rows * C(n-1,2) - raw / 2.  b, a < 2^31.
// EXTRA = false drops the j = 3 accumulator, the rank output and the row groups (the common call) at compile time.
template <bool EXTRA>
__device__ __forceinline__ void emit_rank(const RankOut &o, i64 row_global, i64 acc_off, u32 c, u32 b, u32 a) {
    if (!EXTRA || o.raw2)  // rank-only calls (no accumulator) skip the RED
        atomicAdd((unsigned long long *)&o.raw2[acc_off + c], (u64)b * (u64)(b - 1u) + (u64)a * (u64)(a - 1u));
    if (EXTRA) {
        if (o.acc3)
            atomicAdd((u64 *)&o.acc3[acc_off + c], (u64)(o.full3 - comb3_dev((i64)b) - comb3_dev((i64)a)));
        if (o.rank_b) {
            o.rank_b[row_global * o.n + c] = (int)b;
            if (o.rank_a) o.rank_a[row_global * o.n + c] = (int)a;
        }
    }
}

// count = number of accumulator entries (n per group)
__global__ void mbd_finish_kernel(const u64 *__restrict__ raw2, i64 *__restrict__ acc2, const i64 count,
                                  const i64 rows_full2, const int accumulate) {
    const i64 c = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (c < count) {
        const i64 v = rows_full2 - (i64)(raw2[c] >> 1);
        acc2[c] = accumulate ? acc2[c] + v : v;  // a fresh result needs no zeroing pass
    }
}

// Runs of equal 22-bit keys in a sorted part (collisions of distinct values, or true ties).  The caller has
// published the sorted keys (position pos = lane*EPL + i at skeys[i*32 + lane]) and zeroed sflag.  Every
// position finds its run start with a max-scan over head positions; the run's last element records the run
// length and every element that differs from the run's first value flags the run.  A run of one repeated
// value (tie-heavy data; any length) then costs O(1) per element; only a run that mixes distinct values
// under one key is counted pairwise.  The part lists hold float offsets, so the EXACT values are read from
// the row of X through the curve ids.  Kept out of line: it is rare and must not cost the sort registers.
// LINEAR: the sorted keys lie at skeys[pos] (sub-bin ranking) instead of the register-blocked layout.
template <int EPL, bool LINEAR>
__device__ __forceinline__ int run_at(const int pos) {
    return LINEAR ? pos : (pos % EPL) * 32 + pos / EPL;
}

template <int EPL, bool LINEAR = false>
__device__ __noinline__ void resolve_runs(const double *__restrict__ xrow, const u32 *__restrict__ pj, const int cnt,
                                          const u32 *skeys, u32 *sres, u32 *sflag, const int lane) {
    const int p0 = lane * EPL;
    const u32 r_before = p0 > 0 && p0 <= cnt ? skeys[run_at<EPL, LINEAR>(p0 - 1)] >> 10 : 0xffffffffu;
    int last_head = -1;  // last run start inside this lane's chunk
    u32 rp = r_before;
#pragma unroll 1
    for (int i = 0; i < EPL && p0 + i < cnt; ++i) {
        const u32 r = skeys[run_at<EPL, LINEAR>(p0 + i)] >> 10;
        if (r != rp) last_head = p0 + i;
        rp = r;
    }
    int carry = last_head;  // inclusive max-scan over lanes, then shifted by one lane
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int up = __shfl_up_sync(0xffffffffu, carry, d);
        if (lane >= d) carry = max(carry, up);
    }
    carry = __shfl_up_sync(0xffffffffu, carry, 1);
    if (lane == 0) carry = 0;
    int rs = carry;
    rp = r_before;
#pragma unroll 1
    for (int i = 0; i < EPL && p0 + i < cnt; ++i) {
        const int pos = p0 + i;
        const u32 k = skeys[run_at<EPL, LINEAR>(p0 + i)];
        const u32 r = k >> 10;
        if (r != rp) rs = pos;
        rp = r;
        const u32 rn = pos + 1 < cnt ? skeys[run_at<EPL, LINEAR>(pos + 1)] >> 10 : 0xffffffffu;
        u32 mark = rn != r ? (u32)(pos + 1 - rs) : 0u;  // run length, recorded by the run's last element
        if (rs != pos) {
            const u32 k0 = skeys[run_at<EPL, LINEAR>(rs)];
            if (!(xrow[pj[k & 1023u]] == xrow[pj[k0 & 1023u]])) mark |= 0x80000000u;  // the run holds distinct values
        }
        if (mark) atomicOr(&sflag[run_at<EPL, LINEAR>(rs)], mark);
    }
    __syncwarp();
    rs = carry;
    rp = r_before;
#pragma unroll 1
    for (int i = 0; i < EPL && p0 + i < cnt; ++i) {
        const int pos = p0 + i;
        const u32 k = skeys[run_at<EPL, LINEAR>(p0 + i)];
        const u32 r = k >> 10;
        if (r != rp) rs = pos;
        rp = r;
        const u32 f = sflag[run_at<EPL, LINEAR>(rs)];
        const int len = (int)(f & 0x7fffffffu);
        if (len == 1) continue;  // not in a run: written by the caller's fast path
        const int slot = (int)(k & 1023u);
        int less = 0, greater = 0;
        if (f & 0x80000000u) {  // mixed run: exact pairwise counting inside the run
            const double xs = xrow[pj[slot]];
            for (int m = rs; m < rs + len; ++m) {
                const double xm = xrow[pj[skeys[run_at<EPL, LINEAR>(m)] & 1023u]];
                less += xm < xs;
                greater += xm > xs;
            }
        }
        sres[slot] = (u32)(rs + less) | ((u32)(rs + len - greater) << 16);
    }
}

constexpr int EMIT_DEPTH = 4;

// Emission of one ranked part in slot order (coalesced curve ids).  The RED's address waits for its id: a
// one-at-a-time loop spent 40 % of the kernel's stall samples here, so EMIT_DEPTH ids are fetched a step ahead
// (the caller fetched the first group under its sort).
template <bool EXTRA>
__device__ __forceinline__ void emit_part(const u32 *__restrict__ pj, const int cnt, const u32 base,
                                          const i64 row_global, const RankOut &o, const u32 *sres, const int lane,
                                          u32 (&jnext)[EMIT_DEPTH]) {
    const u32 n32 = (u32)o.n;
    const i64 acc_off = EXTRA ? acc_offset(o, row_global) : 0;  // grouped calls take the EXTRA instantiation
#pragma unroll 1
    for (int s0 = lane; s0 < cnt; s0 += 32 * EMIT_DEPTH) {
        u32 j[EMIT_DEPTH], res[EMIT_DEPTH];
#pragma unroll
        for (int u = 0; u < EMIT_DEPTH; ++u) {
            j[u] = jnext[u];
            const int s = s0 + 32 * u;
            res[u] = s < cnt ? sres[s] : 0u;
            const int sn = s + 32 * EMIT_DEPTH;
            jnext[u] = sn < cnt ? pj[sn] : 0u;
        }
#pragma unroll
        for (int u = 0; u < EMIT_DEPTH; ++u)
            if (s0 + 32 * u < cnt)
                emit_rank<EXTRA>(o, row_global, acc_off, j[u], base + (res[u] & 0xffffu), n32 - base - (res[u] >> 16));
    }
    __syncwarp();
}

// skeys / sres / sflag: this warp's shared scratch (CAP words each).
// px: the part's values as float offsets from its reference splitter (monotone in x; equal offsets do NOT imply
// equal values, so everything that shares a key is resolved on the exact values).  [lo, hi): range of the
// offsets when it is known from the splitters (interior parts); otherwise (first / last part, single-part
// rows) have_range is false and the range is measured.
template <int EPL, bool EXTRA>
__device__ __forceinline__ void rank_part(const float *__restrict__ px, const u32 *__restrict__ pj,
                                          const double *__restrict__ xrow, const int cnt, const u32 base,
                                          const i64 row_global, const RankOut &o, u32 *skeys, u32 *sres, u32 *sflag,
                                          const int lane, float lo, float hi, const bool have_range) {
    if (!have_range) {
        lo = INFINITY;
        hi = -INFINITY;
#pragma unroll 1
        for (int s = lane; s < cnt; s += 32) {
            const float x = px[s];
            lo = fminf(lo, x);
            hi = fmaxf(hi, x);
        }
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            lo = fminf(lo, __shfl_xor_sync(0xffffffffu, lo, d));
            hi = fmaxf(hi, __shfl_xor_sync(0xffffffffu, hi, d));
        }
    }
    // monotone 22-bit key | slot id: every step below is monotone in the offset, hence in x.  hi == lo gives
    // scale = inf and one key for all (0 * inf = NaN converts to 0): one run, resolved exactly.
    const float scale = (float)KEY_MAX / (hi - lo);
    u32 jnext[EMIT_DEPTH];  // curve ids of the first emission group, fetched under the sort
#pragma unroll
    for (int u = 0; u < EMIT_DEPTH; ++u) jnext[u] = lane + 32 * u < cnt ? pj[lane + 32 * u] : 0u;
    u32 v[EPL];
#pragma unroll
    for (int k = 0; k < EPL; ++k) {
        const int s = lane + 32 * k;
        u32 key = 0xffffffffu;
        if (s < cnt) {
            const u32 r = min((u32)__float2uint_rz((px[s] - lo) * scale), KEY_MAX);  // negative / NaN -> 0
            key = (r << 10) | (u32)s;
        }
        v[k] = key;
    }
    warp_bitonic_sort<EPL, u32>(v, lane);

    // equal-key neighbours (collisions of distinct values or true ties) are rare: detect them on registers
    const u32 prev_lane = __shfl_up_sync(0xffffffffu, v[EPL - 1], 1);
    const u32 next_lane = __shfl_down_sync(0xffffffffu, v[0], 1);
    bool any_run = false;
#pragma unroll
    for (int i = 0; i < EPL; ++i) {
        const int pos = lane * EPL + i;
        const u32 r = v[i] >> 10;
        const u32 kl = i > 0 ? v[i - 1] : prev_lane;
        const u32 kr = i + 1 < EPL ? v[i + 1] : next_lane;
        const bool left = pos > 0 && (kl >> 10) == r;
        const bool right = pos + 1 < cnt && (kr >> 10) == r;
        const bool in_run = pos < cnt && (left || right);
        any_run |= in_run;
        if (pos < cnt && !in_run) sres[v[i] & 1023u] = (u32)pos | ((u32)(pos + 1) << 16);
    }
    if (__any_sync(0xffffffffu, any_run)) {
#pragma unroll
        for (int i = 0; i < EPL; ++i) {
            skeys[i * 32 + lane] = v[i];
            sflag[i * 32 + lane] = 0u;
        }
        __syncwarp();
        resolve_runs<EPL>(xrow, pj, cnt, skeys, sres, sflag, lane);
    }
    __syncwarp();
    emit_part<EXTRA>(pj, cnt, base, row_global, o, sres, lane, jnext);
}

// ---------------------------------------------------------------------------------------------
// 3a. sub-bin ranking of a part of at most CAP/2 values (the common case): instead of a 512-wide sorting
//     network over the warp (45 stages, 15 of them shuffles: 56 % of the old rank kernel's instructions),
//     the 22-bit keys are counted into 64 (128 for parts of 513..1024 values) equal-width sub-bins of the part's range (the part spans one
//     1/P quantile of the row, so its density is nearly flat and a bin holds cnt/64 +- a few values), a
//     warp scan turns the counts into bin starts, the keys are scattered to their bins in shared memory, and
//     every LANE sorts its two (four) whole bins of at most SB_CAP keys on its own registers with a 60-comparator
//     network -- no shuffles, no selects, no padding of the part to a power of two.  Equal keys always share a
//     bin, so runs (collisions / ties) are found by the sorting lane and resolved as before.  A part in which a
//     bin overflows (tail parts with a decaying density, heavy ties) is handed to the work list of
//     mbd_rank_big_kernel, whose full sorting network ranks any part.
// ---------------------------------------------------------------------------------------------
constexpr int SB_CAP = 16;    // keys one lane sorts per bin
// EPL keys per lane when loading (16: parts of up to 512 values, 32: up to 1024); EPL / 8 bins per lane, so a
// bin holds a quarter of its capacity on average when the part is full
template <int EPL> struct SubBin {
    static constexpr int BPL = EPL / 8;           // bins per lane (2 or 4)
    static constexpr int BINS = 32 * BPL;         // 64 or 128
    static constexpr int SHIFT = EPL == 16 ? 26 : 25;  // packed key >> SHIFT = bin (22 key bits above 10 slot bits)
};
static_assert(KEY_BITS == 22, "SubBin::SHIFT assumes 22-bit keys over 10 slot bits");

// One lane sorts bin [start, start + c) of skeys on its registers and records the final position of every key that
// shares its 22-bit key with no neighbour (sres[slot] = pos | (pos + 1) << 16); returns whether a run of equal keys
// was seen.  WRITEBACK stores the sorted keys for resolve_runs (second pass, only when the warp saw a run).
template <bool WRITEBACK>
__device__ __forceinline__ bool subbin_sort_bin(u32 *skeys, u32 *sres, const int start, const int c) {
    u32 w[SB_CAP];
#pragma unroll
    for (int i = 0; i < SB_CAP; ++i) w[i] = i < c ? skeys[start + i] : 0xffffffffu;
    thread_sort16<u32>(w);
    bool any_run = false;
    bool eq_prev = false;  // w[i-1] and w[i] share their 22-bit key
#pragma unroll
    for (int i = 0; i < SB_CAP; ++i) {
        const bool eq_next = i + 1 < SB_CAP && i + 1 < c && ((w[i] ^ w[i + 1 < SB_CAP ? i + 1 : i]) < 1024u);
        const bool live = i < c;
        if (WRITEBACK) {
            if (live) skeys[start + i] = w[i];
        } else {
            const bool in_run = eq_prev || eq_next;
            any_run |= in_run;
            if (live && !in_run) sres[w[i] & 1023u] = (u32)(start + i) * 0x10001u + 0x10000u;
        }
        eq_prev = eq_next;
    }
    return any_run;
}

// bin b of this lane starts at start0 + (counts of the lane's earlier bins, packed one byte each in cpack)
__device__ __forceinline__ int subbin_start(const int start0, const u32 cpack, const int b) {
    int s = start0;
#pragma unroll
    for (int k = 0; k < 4; ++k)
        if (k < b) s += (int)((cpack >> (8 * k)) & 255u);
    return s;
}

template <int EPL>
__device__ __noinline__ void subbin_resolve(const double *__restrict__ xrow, const u32 *__restrict__ pj, const int cnt,
                                            u32 *skeys, u32 *sres, u32 *sflag, const int lane, const int start0,
                                            const u32 cpack) {
#pragma unroll 1
    for (int b = 0; b < SubBin<EPL>::BPL; ++b)
        subbin_sort_bin<true>(skeys, sres, subbin_start(start0, cpack, b), (int)((cpack >> (8 * b)) & 255u));
    __syncwarp();
#pragma unroll
    for (int k = 0; k < EPL; ++k) sflag[lane + 32 * k] = 0u;
    __syncwarp();
    resolve_runs<EPL, true>(xrow, pj, cnt, skeys, sres, sflag, lane);
}

// returns false (warp-uniform, nothing emitted) when a bin holds more than SB_CAP keys
template <int EPL, bool EXTRA>
__device__ __forceinline__ bool rank_part_subbin(const float *__restrict__ px, const u32 *__restrict__ pj,
                                                 const double *__restrict__ xrow, const int cnt, const u32 base,
                                                 const i64 row_global, const RankOut &o, u32 *skeys, u32 *sres,
                                                 u32 *sflag, const int lane, float lo, float hi,
                                                 const bool have_range) {
    typedef SubBin<EPL> SB;
    u32 *hist = sflag;  // [BINS] counts, then bin cursors (sflag proper is only needed by resolve_runs)
#pragma unroll
    for (int b = 0; b < SB::BPL; ++b) hist[lane + 32 * b] = 0u;
    // all loads of the part first: an atomic between two loads would serialise their latencies
    float xv[EPL];
#pragma unroll
    for (int k = 0; k < EPL; ++k) xv[k] = lane + 32 * k < cnt ? px[lane + 32 * k] : 0.f;
    u32 jnext[EMIT_DEPTH];
#pragma unroll
    for (int u = 0; u < EMIT_DEPTH; ++u) jnext[u] = lane + 32 * u < cnt ? pj[lane + 32 * u] : 0u;
    if (!have_range) {
        lo = INFINITY;
        hi = -INFINITY;
#pragma unroll
        for (int k = 0; k < EPL; ++k)
            if (lane + 32 * k < cnt) {
                lo = fminf(lo, xv[k]);
                hi = fmaxf(hi, xv[k]);
            }
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            lo = fminf(lo, __shfl_xor_sync(0xffffffffu, lo, d));
            hi = fmaxf(hi, __shfl_xor_sync(0xffffffffu, hi, d));
        }
    }
    const float scale = (float)KEY_MAX / (hi - lo);  // see rank_part
    __syncwarp();
    u32 v[EPL];
#pragma unroll
    for (int k = 0; k < EPL; ++k) {
        const int s = lane + 32 * k;
        u32 key = 0xffffffffu;
        if (s < cnt) {
            const u32 r = min((u32)__float2uint_rz((xv[k] - lo) * scale), KEY_MAX);
            key = (r << 10) | (u32)s;
            atomicAdd(&hist[key >> SB::SHIFT], 1u);
        }
        v[k] = key;
    }
    __syncwarp();
    u32 cpack = 0u, tot = 0u;  // this lane's bin counts, one byte each
    bool over = false;
#pragma unroll
    for (int b = 0; b < SB::BPL; ++b) {
        const u32 c = hist[SB::BPL * lane + b];
        over |= c > (u32)SB_CAP;
        cpack |= min(c, 255u) << (8 * b);
        tot += c;
    }
    if (__any_sync(0xffffffffu, over)) return false;
    u32 incl = tot;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const u32 up = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += up;
    }
    const int start0 = (int)(incl - tot);  // first sorted position of this lane's bins
    __syncwarp();
#pragma unroll
    for (int b = 0; b < SB::BPL; ++b) hist[SB::BPL * lane + b] = (u32)subbin_start(start0, cpack, b);
    __syncwarp();
#pragma unroll
    for (int k = 0; k < EPL; ++k)
        if (v[k] != 0xffffffffu) skeys[atomicAdd(&hist[v[k] >> SB::SHIFT], 1u)] = v[k];  // any order inside the bin
    __syncwarp();
    bool any_run = false;
#pragma unroll 1
    for (int b = 0; b < SB::BPL; ++b)  // rolled: one copy of the 60-comparator network in the instruction cache
        any_run |= subbin_sort_bin<false>(skeys, sres, subbin_start(start0, cpack, b), (int)((cpack >> (8 * b)) & 255u));
    if (__any_sync(0xffffffffu, any_run))  // rare: publish the sorted keys and resolve the runs exactly
        subbin_resolve<EPL>(xrow, pj, cnt, skeys, sres, sflag, lane, start0, cpack);
    __syncwarp();
    emit_part<EXTRA>(pj, cnt, base, row_global, o, sres, lane, jnext);
    return true;
}

constexpr int RANK_WARPS = 4;

// One warp per (row, part).  Two instantiations share the work by part size so that the common case
// (<= 512 values, 8 or 16 keys per lane) is not held to the register and shared-memory budget of the
// rare 1024-value case: BIG = false ranks parts with cnt <= 512, BIG = true the others.
struct RankArgs {
    int P;
    const int *cursor;         // [rows][P] fill counts
    const u32 *pbase;          // [rows][P] exclusive prefix of the fill counts (#values in lower parts)
    const int *rowflag;        // [rows] bit 0: has parts with > CAP values (all-equal classes), bit 1: generic path,
                               //        bit 2: tie-heavy sample (skip the sub-bin attempt)
    const float *splitters_f;  // [rows][P-1] offsets from the row's reference
    const float *part_x;       // [rows][row_stride] offsets from the part's reference splitter
    const u32 *part_j;         // [rows][row_stride] curve ids
    const double *X;           // the rows of this block (exact values for run resolution)
    i64 ld;
    i64 row_stride, row0;
    const int *only;           // masked call: rows are ranked only if only[row] & 2 (null: all rows)
    int2 *biglist;             // (row, part) of parts with more than CAP/2 values
    int *bigcount;             // [0] entries appended, [1] entries claimed
};

template <int EPL, bool EXTRA>
__device__ __forceinline__ void rank_one(const RankArgs &a, const RankOut &o, const i64 row, const int part,
                                         const int cnt, u32 *skeys, u32 *sres, u32 *sflag, const int lane) {
    const int P = a.P;
    const u32 base = a.pbase[row * P + part];
    // interior parts: the offsets lie in [0, splitter[part] - splitter[part-1])
    const bool have_range = part > 0 && part < P - 1;
    float hi = 0.f;
    if (have_range) {
        const float *sp = a.splitters_f + row * (P - 1);
        hi = (float)((double)sp[part] - (double)sp[part - 1]);
    }
    const float *px = a.part_x + row * a.row_stride + (i64)part * CAP;
    const u32 *pj = a.part_j + row * a.row_stride + (i64)part * CAP;
    rank_part<EPL, EXTRA>(px, pj, a.X + row * a.ld, cnt, base, a.row0 + row, o, skeys, sres, sflag, lane, 0.f, hi,
                          have_range);
}

// One warp per (row, part) for parts of at most CAP/2 values (8 or 16 keys per lane, 56 registers);
// bigger parts are appended to a work list for mbd_rank_big_kernel so that the common case is not held
// to the register / shared-memory budget of the rare 1024-value case.
template <bool EXTRA>
__global__ void __launch_bounds__(RANK_WARPS * 32, 8) mbd_rank_kernel(const RankArgs a, const RankOut o) {
    __shared__ u32 s_keys[RANK_WARPS][CAP / 2];
    __shared__ u32 s_res[RANK_WARPS][CAP / 2];
    __shared__ u32 s_flag[RANK_WARPS][CAP / 2];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const i64 row = blockIdx.y;  // grid: (parts / RANK_WARPS, rows)
    const int part = blockIdx.x * RANK_WARPS + wid;
    if (part >= a.P) return;
    if (a.only && !(a.only[row] & 2)) return;
    if (a.rowflag[row] & 2) return;  // the whole row goes to the generic path
    const int cnt = a.cursor[row * a.P + part];
    if (cnt == 0 || cnt > CAP) return;  // heavy parts (one value repeated > CAP times): mbd_heavy_kernel
    if (cnt > CAP / 2) {
        if (lane == 0) a.biglist[atomicAdd(&a.bigcount[0], 1)] = make_int2((int)row, part);
        return;
    }
    if (cnt <= 256) rank_one<8, EXTRA>(a, o, row, part, cnt, s_keys[wid], s_res[wid], s_flag[wid], lane);
    else rank_one<16, EXTRA>(a, o, row, part, cnt, s_keys[wid], s_res[wid], s_flag[wid], lane);
}

// Sub-bin ranking of the parts of at most 512 values (the main rank kernel): ONE atomic pass -- the arrival
// position returned by the count is the key's place inside its bin's row of SB_CAP slots (row pitch 17 words, so that
// "slot i of every lane's bin" spreads over the banks) -- instead of count, scan and a second atomic pass
// (rank_part_subbin, still used for the 513..1024-value parts); no resolve path either: a part with equal 22-bit keys
// (2 % of the parts on tie-free data) is left to the work list.  1.539 -> 1.513 ms per cfg2 step, 2320 -> 1336 SASS
// instructions.
constexpr int SBF_PITCH = SB_CAP + 1;
template <bool EXTRA>
__device__ __forceinline__ bool rank_part_subbin_fixed(const float *__restrict__ px, const u32 *__restrict__ pj,
                                                       const int cnt, const u32 base, const i64 row_global,
                                                       const RankOut &o, u32 *slots, u32 *hist, u32 *sres, const int lane,
                                                       float lo, float hi, const bool have_range) {
    hist[lane] = 0u;
    hist[lane + 32] = 0u;
    float xv[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) xv[k] = lane + 32 * k < cnt ? px[lane + 32 * k] : 0.f;
    u32 jnext[EMIT_DEPTH];
#pragma unroll
    for (int u = 0; u < EMIT_DEPTH; ++u) jnext[u] = lane + 32 * u < cnt ? pj[lane + 32 * u] : 0u;
    if (!have_range) {
        lo = INFINITY;
        hi = -INFINITY;
#pragma unroll
        for (int k = 0; k < 16; ++k)
            if (lane + 32 * k < cnt) {
                lo = fminf(lo, xv[k]);
                hi = fmaxf(hi, xv[k]);
            }
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            lo = fminf(lo, __shfl_xor_sync(0xffffffffu, lo, d));
            hi = fmaxf(hi, __shfl_xor_sync(0xffffffffu, hi, d));
        }
    }
    const float scale = (float)KEY_MAX / (hi - lo);
    __syncwarp();
#pragma unroll
    for (int k = 0; k < 16; ++k) {
        const int s = lane + 32 * k;
        if (s < cnt) {
            const u32 r = min((u32)__float2uint_rz((xv[k] - lo) * scale), KEY_MAX);
            const u32 bin = r >> (KEY_BITS - 6);
            const u32 pos = atomicAdd(&hist[bin], 1u);
            if (pos < (u32)SB_CAP) slots[bin * SBF_PITCH + pos] = (r << 10) | (u32)s;
        }
    }
    __syncwarp();
    const u32 c0 = hist[2 * lane], c1 = hist[2 * lane + 1];
    if (__any_sync(0xffffffffu, c0 > (u32)SB_CAP || c1 > (u32)SB_CAP)) return false;
    u32 incl = c0 + c1;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const u32 up = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += up;
    }
    const int start0 = (int)(incl - c0 - c1);
    bool any_run = false;
#pragma unroll 1
    for (int h = 0; h < 2; ++h) {
        const int c = (int)(h ? c1 : c0), start = h ? start0 + (int)c0 : start0;
        const u32 *row = slots + (2 * lane + h) * SBF_PITCH;
        u32 w[SB_CAP];
#pragma unroll
        for (int i = 0; i < SB_CAP; ++i) w[i] = i < c ? row[i] : 0xffffffffu;
        thread_sort16<u32>(w);
        bool eq_prev = false;
#pragma unroll
        for (int i = 0; i < SB_CAP; ++i) {
            const bool eq_next = i + 1 < SB_CAP && i + 1 < c && ((w[i] ^ w[i + 1 < SB_CAP ? i + 1 : i]) < 1024u);
            any_run |= eq_prev || eq_next;
            if (i < c) sres[w[i] & 1023u] = (u32)(start + i) * 0x10001u + 0x10000u;
            eq_prev = eq_next;
        }
    }
    if (__any_sync(0xffffffffu, any_run)) return false;  // equal keys: exact resolution on the work list
    __syncwarp();
    emit_part<EXTRA>(pj, cnt, base, row_global, o, sres, lane, jnext);
    return true;
}

// Same grid, sub-bin ranking (3a); parts it cannot rank (a bin overflows) join the big parts on the work list.
template <bool EXTRA>
__global__ void __launch_bounds__(RANK_WARPS * 32, 8) mbd_rank_subbin_kernel(const RankArgs a, const RankOut o) {
    __shared__ u32 s_slots[RANK_WARPS][SB_CAP * 4 * SBF_PITCH];  // 64 bins x 17 words
    __shared__ u32 s_hist[RANK_WARPS][64];
    __shared__ u32 s_res[RANK_WARPS][CAP / 2];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const i64 row = blockIdx.y;
    const int part = blockIdx.x * RANK_WARPS + wid;
    if (part >= a.P) return;
    if (a.only && !(a.only[row] & 2)) return;
    const int flag = a.rowflag[row];
    if (flag & 2) return;
    const int cnt = a.cursor[row * a.P + part];
    if (cnt == 0 || cnt > CAP) return;
    bool done = false;
    if (cnt <= CAP / 2 && !(flag & 4)) {  // bit 2: tie-heavy row (mbd_splitters_kernel), not worth the attempt
        const int P = a.P;
        const u32 base = a.pbase[row * P + part];
        const bool have_range = part > 0 && part < P - 1;
        float hi = 0.f;
        if (have_range) {
            const float *sp = a.splitters_f + row * (P - 1);
            hi = (float)((double)sp[part] - (double)sp[part - 1]);
        }
        const float *px = a.part_x + row * a.row_stride + (i64)part * CAP;
        const u32 *pj = a.part_j + row * a.row_stride + (i64)part * CAP;
        done = rank_part_subbin_fixed<EXTRA>(px, pj, cnt, base, a.row0 + row, o, s_slots[wid], s_hist[wid], s_res[wid],
                                             lane, 0.f, hi, have_range);
    }
    if (!done && lane == 0) a.biglist[atomicAdd(&a.bigcount[0], 1)] = make_int2((int)row, part);
}

// persistent: warps claim entries of the work list -- parts of 513..1024 values (sub-bin ranking with 128 bins
// when `subbin`, the full sorting network otherwise or when a bin overflows) and the parts of at most 512 values
// whose sub-bin ranking overflowed (sorting network).
// The overflowed parts of at most 512 values need only the small network (64 registers, 6 KB of shared memory per
// warp): they get their own persistent kernel at full occupancy instead of waiting in the big-part kernel, whose
// 128 registers and 12 KB per warp leave 16 warps per SM (one kernel for both: 162 us of a 1.56 ms step).
template <bool EXTRA>
__global__ void __launch_bounds__(RANK_WARPS * 32, 8) mbd_rank_overflow_kernel(const RankArgs a, const RankOut o) {
    __shared__ u32 s_keys[RANK_WARPS][CAP / 2];
    __shared__ u32 s_res[RANK_WARPS][CAP / 2];
    __shared__ u32 s_flag[RANK_WARPS][CAP / 2];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int total = a.bigcount[0];
    for (;;) {
        int i = 0;
        if (lane == 0) i = atomicAdd(&a.bigcount[3], 1);
        i = __shfl_sync(0xffffffffu, i, 0);
        if (i >= total) break;
        const int2 e = a.biglist[i];
        const int cnt = a.cursor[(i64)e.x * a.P + e.y];
        if (cnt > CAP / 2) continue;  // the big-part kernel's
        if (cnt <= 256) rank_one<8, EXTRA>(a, o, (i64)e.x, e.y, cnt, s_keys[wid], s_res[wid], s_flag[wid], lane);
        else rank_one<16, EXTRA>(a, o, (i64)e.x, e.y, cnt, s_keys[wid], s_res[wid], s_flag[wid], lane);
    }
}

template <bool EXTRA>
__global__ void __launch_bounds__(RANK_WARPS * 32, 4) mbd_rank_big_kernel(const RankArgs a, const RankOut o,
                                                                          const int subbin) {
    __shared__ u32 s_keys[RANK_WARPS][CAP];
    __shared__ u32 s_res[RANK_WARPS][CAP];
    __shared__ u32 s_flag[RANK_WARPS][CAP];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int total = a.bigcount[0];
    for (;;) {
        int i = 0;
        if (lane == 0) i = atomicAdd(&a.bigcount[1], 1);
        i = __shfl_sync(0xffffffffu, i, 0);
        if (i >= total) break;
        const int2 e = a.biglist[i];
        const i64 row = e.x;
        const int part = e.y, cnt = a.cursor[row * a.P + part];
        if (cnt <= CAP / 2) {
            if (subbin == 2) continue;  // overflowed small parts have their own kernel (mbd_rank_overflow_kernel)
            rank_one<16, EXTRA>(a, o, row, part, cnt, s_keys[wid], s_res[wid], s_flag[wid], lane);
            continue;
        }
        bool done = false;
        if (subbin && !(a.rowflag[row] & 4)) {
            const int P = a.P;
            const bool have_range = part > 0 && part < P - 1;
            float hi = 0.f;
            if (have_range) {
                const float *sp = a.splitters_f + row * (P - 1);
                hi = (float)((double)sp[part] - (double)sp[part - 1]);
            }
            done = rank_part_subbin<32, EXTRA>(a.part_x + row * a.row_stride + (i64)part * CAP,
                                               a.part_j + row * a.row_stride + (i64)part * CAP, a.X + row * a.ld, cnt,
                                               a.pbase[row * P + part], a.row0 + row, o, s_keys[wid], s_res[wid],
                                               s_flag[wid], lane, 0.f, hi, have_range);
        }
        if (!done) rank_one<32, EXTRA>(a, o, row, part, cnt, s_keys[wid], s_res[wid], s_flag[wid], lane);
    }
}

// ---------------------------------------------------------------------------------------------
// 3b. heavy parts: a part with more than CAP values can only arise when few VALUES are repeated very often
//     (equal values always share a part; distinct values are spread by the equal-mass splitters).  Such a
//     part needs no sorting.  One CTA per row, run BEFORE the rank kernels; it first writes the row's
//     exclusive prefix of part sizes (pbase) for them, and rows without heavy parts stop there.  Otherwise:
//       pass 1  every value of a heavy part is entered in the part's table of at most HV_VALUES distinct
//               values (shared memory) and counted; a part with more distinct values, or more than HV_PARTS
//               heavy parts, hands the whole row to the generic path (bit 1) and nothing is emitted;
//       pass 2  each member gets b = #values in lower parts + #smaller values of its part, a likewise.
//     Members are found by re-running the part lookup on the row (the part lists only keep CAP values).
// ---------------------------------------------------------------------------------------------
constexpr int HV_PARTS = 128;
constexpr int HV_VALUES = 8;
constexpr int HV_THREADS = 1024;
constexpr int HV_UNROLL = 4;
constexpr u64 HV_EMPTY = ~0ull;  // a NaN pattern: never equals the canonical bits of a finite value

__device__ __forceinline__ int hv_find(const volatile u64 *tab, const u64 bits) {
#pragma unroll
    for (int k = 0; k < HV_VALUES; ++k)
        if (tab[k] == bits) return k;
    return -1;
}

__global__ void __launch_bounds__(HV_THREADS) mbd_heavy_kernel(const double *__restrict__ X, const i64 n, const i64 ld,
                                                        const int P, const float *__restrict__ splitters_f,
                                                        const unsigned short *__restrict__ tables,
                                                        const int *__restrict__ cursor, int *__restrict__ rowflag,
                                                        u32 *__restrict__ pbase, const i64 row0, const RankOut o,
                                                        const int *__restrict__ only) {
    if (only && !(only[blockIdx.x] & 2)) return;
    __shared__ float splf[MAX_PARTS + SPL_PAD];
    __shared__ unsigned short tbl[PT_BUCKETS];
    __shared__ int cnt[MAX_PARTS];
    __shared__ u32 base[MAX_PARTS];
    __shared__ short hidx[MAX_PARTS];
    __shared__ u64 tab[HV_PARTS][HV_VALUES];
    __shared__ int tcnt[HV_PARTS][HV_VALUES];
    __shared__ int tbelow[HV_PARTS][HV_VALUES];
    __shared__ int s_bad, s_heavy;
    __shared__ u32 s_wsum[HV_THREADS / 32];
    const int row = blockIdx.x, tid = threadIdx.x;
    // every row: exclusive prefix of the part sizes (#values in lower parts) for the rank kernels
    const u32 mycnt = tid < P ? (u32)cursor[(i64)row * P + tid] : 0u;
    u32 incl = mycnt;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const u32 up = __shfl_up_sync(0xffffffffu, incl, d);
        if ((tid & 31) >= d) incl += up;
    }
    if ((tid & 31) == 31) s_wsum[tid >> 5] = incl;
    __syncthreads();
    if (tid < 32) {
        const u32 t = tid < (int)(blockDim.x >> 5) ? s_wsum[tid] : 0u;
        u32 ws = t;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const u32 up = __shfl_up_sync(0xffffffffu, ws, d);
            if (tid >= d) ws += up;
        }
        s_wsum[tid] = ws - t;
    }
    __syncthreads();
    const u32 mybase = incl - mycnt + s_wsum[tid >> 5];
    if (tid < P) pbase[(i64)row * P + tid] = mybase;
    if ((rowflag[row] & 3) != 1) return;  // no heavy part, or already generic
    const int nspl = P - 1;
    const double *xr = X + (i64)row * ld;
    const double x0 = row_reference(xr, n);
    fill_splitters(splf, splitters_f + (i64)row * nspl, nspl, tid, blockDim.x);
    for (int b = tid; b < PT_BUCKETS; b += blockDim.x) tbl[b] = nspl > 0 ? tables[(i64)row * PT_BUCKETS + b] : 0;
    if (tid < P) {
        cnt[tid] = (int)mycnt;
        base[tid] = mybase;
    }
    for (int i = tid; i < HV_PARTS * HV_VALUES; i += blockDim.x) {
        (&tab[0][0])[i] = HV_EMPTY;
        (&tcnt[0][0])[i] = 0;
    }
    __syncthreads();
    if (tid == 0) {  // P <= 1024 and only rows with heavy parts get here: a serial pass is cheap
        int heavy = 0;
        for (int p = 0; p < P; ++p) {
            hidx[p] = -1;
            if (cnt[p] > CAP) {
                if (heavy < HV_PARTS) hidx[p] = (short)heavy;
                ++heavy;
            }
        }
        s_heavy = heavy;
        s_bad = heavy > HV_PARTS;
    }
    float f_first = 0.f, inv_w = 0.f;
    if (nspl > 0) {
        f_first = splf[1];
        const float w = (splf[nspl] - f_first) * (1.0f / PT_BUCKETS);
        if (w > 0.f && w < INFINITY) inv_w = 1.0f / w;
    }
    __syncthreads();
    if (!s_bad) {
        for (i64 c0 = tid; c0 < n; c0 += (i64)HV_UNROLL * blockDim.x) {
            double xs[HV_UNROLL];  // loads first: the row scan is latency bound with one CTA per row
#pragma unroll
            for (int u = 0; u < HV_UNROLL; ++u) {
                const i64 c = c0 + (i64)u * blockDim.x;
                xs[u] = c < n ? xr[c] : 0.0;
            }
#pragma unroll
            for (int u = 0; u < HV_UNROLL; ++u) {
                if (c0 + (i64)u * blockDim.x >= n) break;
                const double x = xs[u];
                float lower;
                const int part = nspl > 0 ? part_of(__double2float_rn(x - x0), splf, tbl, f_first, inv_w, lower) : 0;
                const int h = hidx[part];
                if (h < 0) continue;
                const u64 bits = (u64)__double_as_longlong(x + 0.0);  // -0.0 and +0.0 are one value
                int k = hv_find(tab[h], bits);
                if (k < 0) {  // not yet entered: claim the first free entry (or meet a racing equal entry)
                    for (k = 0; k < HV_VALUES; ++k) {
                        const u64 old = atomicCAS((unsigned long long *)&tab[h][k], HV_EMPTY, bits);
                        if (old == HV_EMPTY || old == bits) break;
                    }
                    if (k == HV_VALUES) {
                        s_bad = 1;
                        continue;
                    }
                }
                atomicAdd(&tcnt[h][k], 1);
            }
        }
    }
    __syncthreads();
    if (s_bad) {
        if (tid == 0) atomicOr(&rowflag[row], 2);
        return;
    }
    for (int i = tid; i < s_heavy * HV_VALUES; i += blockDim.x) {
        const int h = i / HV_VALUES, k = i % HV_VALUES;
        int below = 0;
        if (tcnt[h][k] > 0) {
            const double vk = __longlong_as_double((long long)tab[h][k]);
            for (int m = 0; m < HV_VALUES; ++m)
                if (tcnt[h][m] > 0 && __longlong_as_double((long long)tab[h][m]) < vk) below += tcnt[h][m];
        }
        tbelow[h][k] = below;
    }
    const i64 acc_off = acc_offset(o, row0 + row);
    __syncthreads();
    for (i64 c0 = tid; c0 < n; c0 += (i64)HV_UNROLL * blockDim.x) {
        double xs[HV_UNROLL];
#pragma unroll
        for (int u = 0; u < HV_UNROLL; ++u) {
            const i64 c = c0 + (i64)u * blockDim.x;
            xs[u] = c < n ? xr[c] : 0.0;
        }
#pragma unroll
        for (int u = 0; u < HV_UNROLL; ++u) {
            const i64 c = c0 + (i64)u * blockDim.x;
            if (c >= n) break;
            const double x = xs[u];
            float lower;
                const int part = nspl > 0 ? part_of(__double2float_rn(x - x0), splf, tbl, f_first, inv_w, lower) : 0;
            const int h = hidx[part];
            if (h < 0) continue;
            const int k = hv_find(tab[h], (u64)__double_as_longlong(x + 0.0));
            const u32 b = base[part] + (u32)tbelow[h][k];
            emit_rank<true>(o, row0 + row, acc_off, (u32)c, b, (u32)n - b - (u32)tcnt[h][k]);
        }
    }
}

// ---------------------------------------------------------------------------------------------
// 4. generic path: one CTA ranks one row (any finite input, any tie structure)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void ce_u64(u64 &a, u64 &b) {
    if (a > b) { const u64 t = a; a = b; b = t; }
}

// sorts tile[0..len) (len power of two <= FB_TILE) ascending; all threads of the CTA participate
__device__ void smem_sort_full(u64 *tile, int len) {
    const int tid = threadIdx.x, nt = blockDim.x;
    for (int k = 2; k <= len; k <<= 1) {
        const int hk = k >> 1;
        for (int i = tid; i < (len >> 1); i += nt) {
            const int blk = i / hk, off = i - blk * hk;
            ce_u64(tile[blk * k + off], tile[blk * k + k - 1 - off]);
        }
        __syncthreads();
        for (int j = k >> 2; j > 0; j >>= 1) {
            for (int i = tid; i < (len >> 1); i += nt) {
                const int a = 2 * j * (i / j) + (i % j);
                ce_u64(tile[a], tile[a + j]);
            }
            __syncthreads();
        }
    }
}

// finishes a merge inside a tile: stages j = len/2 .. 1
__device__ void smem_merge_tail(u64 *tile, int len) {
    const int tid = threadIdx.x, nt = blockDim.x;
    for (int j = len >> 1; j > 0; j >>= 1) {
        for (int i = tid; i < (len >> 1); i += nt) {
            const int a = 2 * j * (i / j) + (i % j);
            ce_u64(tile[a], tile[a + j]);
        }
        __syncthreads();
    }
}

// ranks one row; all threads of the CTA take part
__device__ void fallback_row(const double *__restrict__ X, const i64 n, const i64 ld, const i64 NP, u64 *tile,
                             u64 *__restrict__ scratch, const i64 row_stride, const i64 row0, const RankOut &o,
                             int *__restrict__ status, int *__restrict__ fb_count, const i64 row) {
    const int tid = threadIdx.x, nt = blockDim.x;
    if (tid == 0) atomicAdd(fb_count, 1);
    const double *xr = X + row * ld;
    u64 *keys = scratch + row * row_stride;
    bool bad = false;
    for (i64 c = tid; c < NP; c += nt) {
        u64 k = ~0ull;
        if (c < n) {
            const double x = xr[c];
            bad |= !isfinite(x);
            k = sortable_key(x);
        }
        keys[c] = k;
    }
    if (bad) atomicOr(status, ST_NONFINITE);
    __syncthreads();
    const int tl = NP < FB_TILE ? (int)NP : FB_TILE;
    for (i64 t0 = 0; t0 < NP; t0 += tl) {  // sort every tile in shared memory
        for (int i = tid; i < tl; i += nt) tile[i] = keys[t0 + i];
        __syncthreads();
        smem_sort_full(tile, tl);
        for (int i = tid; i < tl; i += nt) keys[t0 + i] = tile[i];
        __syncthreads();
    }
    for (i64 k = 2 * (i64)tl; k <= NP; k <<= 1) {  // merges wider than a tile: global stages, then tile tails
        const i64 hk = k >> 1;
        for (i64 i = tid; i < (NP >> 1); i += nt) {
            const i64 blk = i / hk, off = i - blk * hk;
            const i64 a = blk * k + off, b = blk * k + k - 1 - off;
            u64 va = keys[a], vb = keys[b];
            if (va > vb) { keys[a] = vb; keys[b] = va; }
        }
        __syncthreads();
        for (i64 j = k >> 2; j >= tl; j >>= 1) {
            for (i64 i = tid; i < (NP >> 1); i += nt) {
                const i64 a = 2 * j * (i / j) + (i % j), b = a + j;
                u64 va = keys[a], vb = keys[b];
                if (va > vb) { keys[a] = vb; keys[b] = va; }
            }
            __syncthreads();
        }
        for (i64 t0 = 0; t0 < NP; t0 += tl) {
            for (int i = tid; i < tl; i += nt) tile[i] = keys[t0 + i];
            __syncthreads();
            smem_merge_tail(tile, tl);
            for (int i = tid; i < tl; i += nt) keys[t0 + i] = tile[i];
            __syncthreads();
        }
    }
    // ranks by binary search in the sorted keys (first n entries are the real ones)
    const i64 acc_off = acc_offset(o, row0 + row);
    for (i64 c = tid; c < n; c += nt) {
        const u64 key = sortable_key(xr[c]);
        i64 lo = 0, hi = n;  // lower bound: first index with keys[idx] >= key
        while (lo < hi) {
            const i64 mid = (lo + hi) >> 1;
            if (keys[mid] < key) lo = mid + 1; else hi = mid;
        }
        const i64 b = lo;
        hi = n;  // upper bound: first index with keys[idx] > key (starts at lo)
        while (lo < hi) {
            const i64 mid = (lo + hi) >> 1;
            if (keys[mid] <= key) lo = mid + 1; else hi = mid;
        }
        emit_rank<true>(o, row0 + row, acc_off, (u32)c, (u32)b, (u32)(n - lo));
    }
}

// persistent over the rows of the block: almost always no row is flagged, and one CTA per row would cost a
// launch of thousands of idle 1024-thread CTAs per call (4-5 % of a call on short rows)
__global__ void __launch_bounds__(1024) mbd_fallback_kernel(const double *__restrict__ X, const i64 n, const i64 ld,
                                                             const i64 NP, const int *__restrict__ rowflag,
                                                             const i64 rows, u64 *__restrict__ scratch,
                                                             const i64 row_stride, const i64 row0, const RankOut o,
                                                             int *__restrict__ status, int *__restrict__ fb_count) {
    __shared__ u64 tile[FB_TILE];
    for (i64 row = blockIdx.x; row < rows; row += gridDim.x) {
        if (!(rowflag[row] & 2)) continue;  // uniform
        fallback_row(X, n, ld, NP, tile, scratch, row_stride, row0, o, status, fb_count, row);
        __syncthreads();
    }
}

__global__ void fill_int_kernel(int *p, i64 count, int value) {
    const i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < count) p[i] = value;
}

}  // namespace sd

#include "mbd_slab.cuh"

namespace sd {

// ---------------------------------------------------------------------------------------------
// driver
// ---------------------------------------------------------------------------------------------
static int pow2ceil_int(i64 v) {
    int p = 1;
    while (p < v) p <<= 1;
    return p;
}

// Geometry of the slab path (mbd_slab.cuh) for rows of n values: the fewest CTAs per row whose entries, bin words
// and bucket table fit one CTA's shared memory.  ok = false: the part pipeline ranks the call.
struct SlabPlan {
    bool ok;
    int G, NBc, NB, ecap, threads;
    size_t smem_rank, smem_hist;
};

static int env_int(const char *name, const int fallback) {
    const char *e = getenv(name);
    return e && *e ? atoi(e) : fallback;
}

static SlabPlan slab_plan(const double *dX, const i64 n, const i64 ld) {
    SlabPlan p;
    memset(&p, 0, sizeof(p));
    if (const char *e = getenv("SD_MBD_PATH"))
        if (!strcmp(e, "parts")) return p;  // A/B aid: the part pipeline everywhere
    i64 min_n = env_int("SD_MBD_SLAB_MIN", (int)SL_MIN_N);
    if (min_n < SL_MIN_N) min_n = SL_MIN_N;  // the hist kernel samples SL_SAMPLE distinct values
    // double2 loads need 16-byte aligned rows; 17-bit curve ids
    if (n < min_n || n > SL_MAX_N || (ld & 1) || ((uintptr_t)dX & 15)) return p;
    int threads = env_int("SD_MBD_SLAB_THREADS", 1024);
    if (threads < 128 || threads > 1024 || (threads & 31)) threads = 1024;
    const int g_forced = env_int("SD_MBD_SLAB_G", 0);
    const i64 nb0 = ceil_div(n, SL_MEAN);
    const size_t smem_max = 232448 - 256;  // 227 KB opt-in limit per CTA, less the kernel's static shared memory
    for (int G = 1; G <= 32; ++G) {
        if (g_forced > 0 && G != g_forced) continue;
        // bins per CTA: a multiple of 1024 (every warp sorts the same number of bins), ~SL_MEAN values per bin
        i64 NBc = ((ceil_div(nb0, G) + 512) / 1024) * 1024;
        if (NBc < 1024) NBc = 1024;
        if (n > NBc * G * (SL_MEAN + 1) + NBc * G / 2) NBc += 1024;  // more than 9.5 per bin
        const i64 per = ceil_div(n, G);
        const i64 ecap = per + per / 16 + 128;  // bins are allotted by the sample's bucket counts: n/G +- a few percent
        if (ecap > 65535 || NBc > 65535) continue;
        const size_t smem = (size_t)(ecap + SL_SORT_CAP) * 4 + (size_t)NBc * 4;
        if (smem > smem_max) continue;
        p.ok = true;
        p.G = G;
        p.NBc = (int)NBc;
        p.NB = (int)(NBc * G);
        p.ecap = (int)ecap;
        p.threads = threads;
        p.smem_rank = smem;
        p.smem_hist = (size_t)p.NB * 4;
        break;
    }
    return p;
}

// The dynamic shared memory the kernels of the rank pipeline may take, set once per context: the slab kernels may
// take all an SM offers beside their static arrays (what a launch takes is its plan's size), so that no call of any
// context on the device lowers a limit another one relies on.
static int mbd_kernel_attributes(sd_ctx *ctx) {
    if (ctx->mbd_attributes_set) return SD_OK;
    int optin = 0;
    SD_CUDA(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, ctx->device));
    SD_CUDA(cudaFuncSetAttribute(mbd_partition_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)PT_SMEM));
    const void *slab[4] = {(const void *)mbd_slab_hist_kernel<SL_HIST_THREADS>, (const void *)mbd_slab_hist_kernel<1024>,
                           (const void *)mbd_slab_rank_kernel<false>, (const void *)mbd_slab_rank_kernel<true>};
    for (const void *f : slab) {
        cudaFuncAttributes fa;
        SD_CUDA(cudaFuncGetAttributes(&fa, f));
        SD_CUDA(cudaFuncSetAttribute(f, cudaFuncAttributeMaxDynamicSharedMemorySize, optin - (int)fa.sharedSizeBytes));
    }
    ctx->mbd_attributes_set = 1;
    return SD_OK;
}

// The part pipeline's geometry and workspaces for one call (blocks of at most Tc rows)
struct PartPlan {
    int P, S;
    i64 NP, row_stride, Tc;
    bool rank_subbin;
    float *part_x, *splitters_f;
    unsigned short *tables;
    u32 *part_j, *pbase;
    int *cursor, *rowflag;
    int2 *biglist;
};

// The slab path on rows [r0, r0 + rows).  Once its rank kernel is queued, *only is the mask of the rows it skipped
// (left to the part pipeline), and *done is set when the host has seen that it skipped none.
static int slab_block(sd_ctx *ctx, const SlabPlan &sp, SlabArgs sa, const SlabReport &rep, const RankOut &o,
                      const bool extra, const double *Xb, const i64 r0, const i64 rows, const int **only, bool *done) {
    cudaStream_t st = ctx->stream;
    sa.X = Xb;
    sa.row0 = r0;
    for (int k = 0; k < 2; ++k)
        if (!ctx->ev_slab[k]) SD_CUDA(cudaEventCreateWithFlags(&ctx->ev_slab[k], cudaEventDisableTiming));
    SD_TRY(prof_begin(ctx, SD_PHASE_MBD_SLAB_HIST));
    mbd_slab_table_kernel<<<(unsigned)rows, SL_TABLE_THREADS, 0, st>>>(sa, rep);
    // Rows this path cannot take are counted twice: after the table kernel (ties, degenerate ranges) and after the
    // hist kernel (a bin, a CTA's share or the pair work over its limit: wild tails, adversarial spreads).  The last
    // CTA of each kernel stores its count into the pinned status mirror (slab_report), so the host decides while later
    // kernels run or are already queued, without leaving the GPU idle.  Many unfit rows after the first count
    // (tie-heavy data) send the whole block to the part pipeline; otherwise the rank kernel skips the flagged rows and
    // the part pipeline ranks just those.
    // A pipelined host call (row blocks copied on a second stream while earlier blocks are ranked) must not stall the
    // host: it skips the counts and always queues the masked part pipeline behind the rank kernel (its CTAs exit at
    // once when no row is flagged: ~50 us per block).  An SD_OPT_ASYNC_DEVICE call does wait: its waits end with the
    // first two kernels, while the rank kernel is still running.
    const bool ask = !ctx->mbd_no_wait;
    if (ask) SD_CUDA(cudaEventRecord(ctx->ev_slab[0], st));
    if (env_int("SD_MBD_SLAB_HIST_THREADS", rows <= (i64)ctx->sm_count ? 1024 : SL_HIST_THREADS) == 1024)
        mbd_slab_hist_kernel<1024><<<(unsigned)rows, 1024, sp.smem_hist, st>>>(sa, rep);
    else
        mbd_slab_hist_kernel<SL_HIST_THREADS><<<(unsigned)rows, SL_HIST_THREADS, sp.smem_hist, st>>>(sa, rep);
    SD_TRY(prof_end(ctx));
    ctx->last.launches += 2;
    const volatile int *counts = ctx->h_status + 2;  // [0] after the hist kernel, [1] after the table kernel
    if (ask) {
        SD_CUDA(cudaEventRecord(ctx->ev_slab[1], st));
        SD_CUDA(cudaEventSynchronize(ctx->ev_slab[0]));
        if ((i64)counts[1] * 16 > rows) return SD_OK;  // all unfit
    }
    const dim3 sgrid((unsigned)sp.G, (unsigned)rows);
    SD_TRY(prof_begin(ctx, SD_PHASE_MBD_SLAB_RANK));
    if (extra) mbd_slab_rank_kernel<true><<<sgrid, sp.threads, sp.smem_rank, st>>>(sa, o);
    else mbd_slab_rank_kernel<false><<<sgrid, sp.threads, sp.smem_rank, st>>>(sa, o);
    SD_TRY(prof_end(ctx));
    ctx->last.launches++;
    *only = sa.rowflag;  // the flagged rows: part pipeline (the generic path costs ~2 ms per long row)
    if (ask) {
        SD_CUDA(cudaEventSynchronize(ctx->ev_slab[1]));  // the rank kernel is queued behind the hist kernel
        *done = counts[0] == 0;
    }
    return SD_OK;
}

// Steps 1-3 of the part pipeline on rows [r0, r0 + rows): all of them, or those the mask `only` flags
template <bool EXTRA>
static int part_block(sd_ctx *ctx, const PartPlan &pp, const RankOut &o, const double *Xb, const i64 ld,
                      const i64 r0, const i64 rows, const int *only) {
    cudaStream_t st = ctx->stream;
    const i64 n = o.n;
    SD_CUDA(cudaMemsetAsync(pp.cursor, 0, (size_t)pp.Tc * (pp.P + 1) * sizeof(int), st));
    if (pp.P > 1) {
        SD_TRY(prof_begin(ctx, SD_PHASE_MBD_SPLITTERS));
        mbd_splitters_kernel<<<(unsigned)rows, SP_THREADS, 0, st>>>(Xb, n, ld, pp.P, pp.S, pp.splitters_f, pp.tables,
                                                                    pp.rowflag, ctx->d_status, only);
        SD_TRY(prof_end(ctx));
        ctx->last.launches++;
    }
    dim3 pgrid((unsigned)ceil_div(n, PT_CHUNK), (unsigned)rows);
    SD_TRY(prof_begin(ctx, SD_PHASE_MBD_PARTITION));
    mbd_partition_kernel<<<pgrid, PT_THREADS, PT_SMEM, st>>>(Xb, n, ld, pp.P, pp.splitters_f, pp.tables, pp.cursor,
                                                             pp.rowflag, pp.part_x, pp.part_j, pp.row_stride,
                                                             ctx->d_status, only);
    SD_TRY(prof_end(ctx));
    ctx->last.launches++;
    SD_TRY(prof_begin(ctx, SD_PHASE_MBD_RANK));
    // rows with parts of more than CAP values (heavy ties): those parts are ranked from value tables
    // one thread per part for the prefix; rows with heavy parts scan their values with the same block
    int hv_threads = 128;
    while (hv_threads < pp.P) hv_threads <<= 1;
    if (n > 16384) hv_threads = HV_THREADS;  // long rows: a heavy row scans n values
    mbd_heavy_kernel<<<(unsigned)rows, hv_threads, 0, st>>>(Xb, n, ld, pp.P, pp.splitters_f, pp.tables, pp.cursor,
                                                            pp.rowflag, pp.pbase, r0, o, only);
    const RankArgs ra = {pp.P,      pp.cursor, pp.pbase,      pp.rowflag, pp.splitters_f, pp.part_x,   pp.part_j,
                         Xb,        ld,        pp.row_stride, r0,         only,           pp.biglist, ctx->d_status + 2};
    SD_CUDA(cudaMemsetAsync(ctx->d_status + 2, 0, 4 * sizeof(int), st));  // appended | claimed (big) | - | claimed (overflow)
    const dim3 rgrid((unsigned)ceil_div(pp.P, RANK_WARPS), (unsigned)rows);
    const unsigned bgrid = (unsigned)(ctx->sm_count * 4);
    const unsigned ogrid = (unsigned)(ctx->sm_count * 8);
    // many parts: the overflowed small parts get their own full-occupancy kernel (-15 us at 256 k parts);
    // few parts (one rank's rows at 8 GPUs): one more persistent launch costs more than it saves (+10 us)
    const bool subbin = pp.rank_subbin, split_overflow = subbin && rows * (i64)pp.P >= 100000;
    if (subbin) mbd_rank_subbin_kernel<EXTRA><<<rgrid, RANK_WARPS * 32, 0, st>>>(ra, o);
    else mbd_rank_kernel<EXTRA><<<rgrid, RANK_WARPS * 32, 0, st>>>(ra, o);
    if (split_overflow) mbd_rank_overflow_kernel<EXTRA><<<ogrid, RANK_WARPS * 32, 0, st>>>(ra, o);
    mbd_rank_big_kernel<EXTRA><<<bgrid, RANK_WARPS * 32, 0, st>>>(ra, o, subbin ? (split_overflow ? 2 : 1) : 0);
    SD_TRY(prof_end(ctx));
    ctx->last.launches += split_overflow ? 4 : 3;
    return SD_OK;
}

// Step 4 on the rows of [r0, r0 + rows) flagged as overflowing, or all of them when forced; idle CTAs exit at once
static int generic_block(sd_ctx *ctx, const PartPlan &pp, const RankOut &o, const double *Xb, const i64 ld,
                         const i64 r0, const i64 rows) {
    if (ctx->mbd_force_fallback) {
        fill_int_kernel<<<(unsigned)ceil_div(rows, 256), 256, 0, ctx->stream>>>(pp.rowflag, rows, 2);
        ctx->last.launches++;
    }
    SD_TRY(prof_begin(ctx, SD_PHASE_MBD_GENERIC));
    const i64 fgrid = rows < 2 * (i64)ctx->sm_count ? rows : 2 * (i64)ctx->sm_count;
    mbd_fallback_kernel<<<(unsigned)fgrid, 1024, 0, ctx->stream>>>(Xb, o.n, ld, pp.NP, pp.rowflag, rows,
                                                                   (u64 *)pp.part_x, pp.NP, r0, o, ctx->d_status,
                                                                   ctx->d_status + 1);
    SD_TRY(prof_end(ctx));
    ctx->last.launches++;
    return SD_OK;
}

// The driver behind mbd_all_device and rank_rows_device; o brings the j = 3 accumulator, rank outputs and row groups.
static int rank_pipeline(sd_ctx *ctx, const double *dX, const i64 T, const i64 n, const i64 ld, i64 *d_acc2,
                         const bool accumulate, RankOut o) {
    if (n < 1 || T < 0 || ld < n) {
        set_error("mbd: bad shape T=%lld n=%lld ld=%lld", (long long)T, (long long)n, (long long)ld);
        return SD_ERR_INVALID;
    }
    if (n >= (1ll << 31)) {
        set_error("mbd: n=%lld exceeds 2^31-1", (long long)n);
        return SD_ERR_UNSUPPORTED;
    }
    const i64 group_rows = o.group_rows;
    if (group_rows < 0 || (group_rows > 0 && T % group_rows != 0)) {
        set_error("mbd: %lld rows are not a multiple of the group size %lld", (long long)T, (long long)group_rows);
        return SD_ERR_INVALID;
    }
    const i64 groups = group_rows > 0 ? T / group_rows : 1;
    const i64 acc_len = n * (groups > 0 ? groups : 1);
    cudaStream_t st = ctx->stream;
    if (!accumulate && d_acc2) {  // d_acc2 itself is WRITTEN by mbd_finish_kernel
        if (o.acc3) SD_CUDA(cudaMemsetAsync(o.acc3, 0, (size_t)acc_len * sizeof(i64), st));
        if (T == 0) SD_CUDA(cudaMemsetAsync(d_acc2, 0, (size_t)acc_len * sizeof(i64), st));
    }
    if (T == 0) return SD_OK;

    int target = TARGET_PART;
    if (const char *e = getenv("SD_MBD_TARGET_PART")) {  // tuning aid
        const int v = atoi(e);
        if (v >= 64 && v <= 512) target = v;
    }
    bool rank_subbin = true;  // SD_MBD_RANK=network selects the warp-wide sorting network (A/B aid)
    if (const char *e = getenv("SD_MBD_RANK")) rank_subbin = strcmp(e, "network") != 0;
    int P = n <= CAP ? 1 : (int)ceil_div(n, target);  // n <= 1024: one part, one warp ranks the whole row
    if (P > MAX_PARTS) P = MAX_PARTS;
    int S = 0;
    if (P > 1) {  // n > 1024 here, so S <= n
        S = pow2ceil_int((i64)OVERSAMPLE * P);
        if (S < 1024) S = 1024;
        if (S > MAX_SAMPLE) S = MAX_SAMPLE;
    }
    const i64 NP = pow2ceil_int(n);
    const i64 row_stride = (i64)P * CAP;  // slots per row in the part lists (4-byte offset + 4-byte curve id)

    // rows per block: keep the part lists within ~6 GB
    const size_t per_row = (size_t)(row_stride > NP ? row_stride : NP) * 8;
    i64 Tc = (i64)((6ull << 30) / per_row);
    if (Tc < 1) Tc = 1;
    if (Tc > T) Tc = T;
    if (Tc > 65535) Tc = 65535;

    // float part lists; the generic path reuses the buffer as NP sortable u64 keys per row
    SD_TRY(ctx->buf[BUF_PART_X].reserve((size_t)Tc * (row_stride * 4 > NP * 8 ? row_stride * 4 : NP * 8)));
    SD_TRY(ctx->buf[BUF_PART_J].reserve((size_t)Tc * row_stride * 4));
    SD_TRY(ctx->buf[BUF_CURSOR].reserve((size_t)Tc * (2 * P + 1) * sizeof(int)));
    SD_TRY(ctx->buf[BUF_SPLIT].reserve((size_t)Tc * (P > 1 ? P - 1 : 1) * sizeof(float) +
                                       (size_t)Tc * PT_BUCKETS * sizeof(unsigned short)));
    float *part_x = ctx->buf[BUF_PART_X].as<float>();
    u32 *part_j = ctx->buf[BUF_PART_J].as<u32>();
    int *cursor = ctx->buf[BUF_CURSOR].as<int>();
    int *rowflag = cursor + (size_t)Tc * P;
    u32 *pbase = reinterpret_cast<u32 *>(rowflag + Tc);
    float *splitters_f = ctx->buf[BUF_SPLIT].as<float>();
    unsigned short *tables = reinterpret_cast<unsigned short *>(splitters_f + (size_t)Tc * (P > 1 ? P - 1 : 1));
    SD_TRY(ctx->buf[BUF_WORK].reserve((size_t)Tc * P * sizeof(int2) + (size_t)acc_len * sizeof(u64)));
    int2 *biglist = ctx->buf[BUF_WORK].as<int2>();
    u64 *raw2 = reinterpret_cast<u64 *>(biglist + (size_t)Tc * P);
    SD_TRY(mbd_kernel_attributes(ctx));

    // slab path (mbd_slab.cuh): per-value codes, bin starts, per-CTA offsets, row flags
    const SlabPlan sp = ctx->mbd_force_fallback ? SlabPlan{} : slab_plan(dX, n, ld);
    // raw2 starts at zero: cleared by the slab path's first table kernel, else by a memset
    SlabReport rep = {ctx->h_status_dev + 2, sp.ok && d_acc2 ? raw2 : nullptr, sp.ok && d_acc2 ? acc_len : 0};
    if (d_acc2 && !sp.ok) SD_CUDA(cudaMemsetAsync(raw2, 0, (size_t)acc_len * sizeof(u64), st));
    SlabArgs sa = {};
    if (sp.ok) {
        const size_t rows_cap = (size_t)Tc;
        const size_t cpitch = (size_t)((n + 3) & ~(i64)3);
        const size_t off_map = rows_cap * cpitch * sizeof(u32);
        const size_t off_tables = off_map + rows_cap * sizeof(double2);
        const size_t off_below = off_tables + rows_cap * SL_BUCKETS * sizeof(uint2);
        const size_t off_flag = off_below + rows_cap * sp.G * sizeof(u32);
        const size_t off_starts = off_flag + rows_cap * sizeof(int);
        SD_TRY(ctx->buf[BUF_SLAB].reserve(off_starts + rows_cap * sp.NB * sizeof(unsigned short)));
        unsigned char *base = ctx->buf[BUF_SLAB].as<unsigned char>();
        sa.n = n;
        sa.ld = ld;
        sa.G = sp.G;
        sa.NBc = sp.NBc;
        sa.ecap = sp.ecap;
        sa.codes = reinterpret_cast<u32 *>(base);
        sa.cpitch = (i64)cpitch;
        sa.rowmap = reinterpret_cast<double2 *>(base + off_map);
        sa.tables = reinterpret_cast<uint2 *>(base + off_tables);
        sa.below = reinterpret_cast<u32 *>(base + off_below);
        sa.rowflag = reinterpret_cast<int *>(base + off_flag);
        sa.starts = reinterpret_cast<unsigned short *>(base + off_starts);
        sa.failcount = ctx->d_status + 6;
        sa.status = ctx->d_status;
    }

    const PartPlan pp = {P, S, NP, row_stride, Tc, rank_subbin, part_x, splitters_f, tables, part_j, pbase, cursor,
                         rowflag, biglist};
    o.raw2 = d_acc2 ? raw2 : nullptr;
    o.n = n;
    o.full2 = (n - 1) * (n - 2) / 2;
    o.full3 = n - 1 < 3 ? 0 : ((n - 1) * (n - 2) / 2) * (n - 3) / 3;
    const bool extra = o.acc3 || o.rank_b || o.group_rows;
    for (i64 r0 = 0; r0 < T; r0 += Tc) {
        const i64 rows = T - r0 < Tc ? T - r0 : Tc;
        const double *Xb = dX + r0 * ld;
        const int *only = nullptr;  // part pipeline restricted to the rows the slab path gave up
        bool done = false;
        if (sp.ok) SD_TRY(slab_block(ctx, sp, sa, rep, o, extra, Xb, r0, rows, &only, &done));
        rep.zero_len = 0;  // later row blocks accumulate
        if (!done && !ctx->mbd_force_fallback)
            SD_TRY(extra ? part_block<true>(ctx, pp, o, Xb, ld, r0, rows, only)
                         : part_block<false>(ctx, pp, o, Xb, ld, r0, rows, only));
        if (!done) SD_TRY(generic_block(ctx, pp, o, Xb, ld, r0, rows));
        SD_CUDA(cudaGetLastError());
    }
    if (d_acc2) {
        mbd_finish_kernel<<<(unsigned)ceil_div(acc_len, 256), 256, 0, st>>>(raw2, d_acc2, acc_len,
                                                                            (group_rows > 0 ? group_rows : T) * o.full2,
                                                                            accumulate ? 1 : 0);
        ctx->last.launches++;
    }
    SD_CUDA(cudaGetLastError());
    return SD_OK;
}

int mbd_all_device(sd_ctx *ctx, const double *dX, i64 T, i64 n, i64 ld, i64 *d_acc2, i64 *d_acc3, bool accumulate,
                   i64 group_rows) {
    RankOut o = {nullptr, d_acc3};
    o.group_rows = group_rows;
    return rank_pipeline(ctx, dX, T, n, ld, d_acc2, accumulate, o);
}

int rank_rows_device(sd_ctx *ctx, const double *dX, i64 T, i64 n, i64 ld, int *d_rank_b, int *d_rank_a) {
    return rank_pipeline(ctx, dX, T, n, ld, nullptr, false, RankOut{nullptr, nullptr, d_rank_b, d_rank_a});
}

constexpr size_t RANK_BLOCK_BUDGET = 1ull << 30;

int rank_block_workspace(sd_ctx *ctx, i64 T, i64 ints_per_row, i64 *RB, int **ws) {
    i64 rb = (i64)(RANK_BLOCK_BUDGET / ((size_t)ints_per_row * sizeof(int)));
    if (rb < 1) rb = 1;
    if (rb > T) rb = T;
    SD_TRY(ctx->buf[BUF_RANKS].reserve((size_t)rb * ints_per_row * sizeof(int)));
    *RB = rb;
    *ws = ctx->buf[BUF_RANKS].as<int>();
    return SD_OK;
}

int for_each_rank_block(sd_ctx *ctx, const double *dX, i64 T, i64 n, i64 ld, bool want_a, i64 max_rows,
                        const RankBlockFn &consume) {
    i64 RB = 0;
    int *rb = nullptr;
    SD_TRY(rank_block_workspace(ctx, T, want_a ? 2 * n : n, &RB, &rb));
    if (RB > max_rows) RB = max_rows;
    int *ra = want_a ? rb + (size_t)RB * n : nullptr;
    for (i64 r0 = 0; r0 < T; r0 += RB) {
        const i64 rows = T - r0 < RB ? T - r0 : RB;
        SD_TRY(rank_rows_device(ctx, dX + r0 * ld, rows, n, ld, rb, ra));
        consume(r0, rows, rb, ra);
        SD_CUDA(cudaGetLastError());
    }
    return SD_OK;
}

}  // namespace sd

extern "C" int sd_mbd_plan(int64_t n, int64_t ld, int64_t *out6) {
    if (!out6 || n < 1 || ld < n) {
        sd::set_error("sd_mbd_plan: bad arguments n=%lld ld=%lld", (long long)n, (long long)ld);
        return SD_ERR_INVALID;
    }
    const sd::SlabPlan p = sd::slab_plan(nullptr, n, ld);
    out6[0] = p.ok ? 1 : 0;
    out6[1] = p.G;
    out6[2] = p.NBc;
    out6[3] = p.ecap;
    out6[4] = (int64_t)p.smem_rank;
    out6[5] = (int64_t)p.smem_hist;
    return SD_OK;
}
