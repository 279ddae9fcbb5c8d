// mbd_slab.cuh -- "slab" form of the K1 rank pipeline (included by mbd.cu; same math, same outputs).
//
// The part pipeline of mbd.cu sends every value through HBM once more (8-byte part-list entries).  Here a row
// never leaves the chip after it has been read:
//
//   mbd_slab_hist_kernel  one CTA per row.  A strided sample of 16384 values gives a trimmed, widened value range
//                         and a 256-bucket estimate of the distribution function over it: a monotone piecewise-linear
//                         map  code(x) = C[k] + frac(x in bucket k) * D[k]  whose integer part is a BIN of ~8 values
//                         and whose next 14 bits order the values inside the bin.  ONE pass over the row then counts
//                         the bins exactly, so that every bin's first position is known -- and every capacity the
//                         rank kernel relies on is VALIDATED -- before a single rank is emitted.  A row that does not
//                         fit (tie-heavy, wild tails) is flagged for the generic path and skipped by all of its rank
//                         CTAs consistently.
//   mbd_slab_rank_kernel  G CTAs per row, CTA g owns bins [g*NBc, (g+1)*NBc): it streams the WHOLE row (its siblings
//                         run beside it, so G-1 of the G reads are L2 hits), keeps the values of its bins as 4-byte
//                         entries (14-bit in-bin key | 17-bit curve id) placed compactly by one shared-memory atomic
//                         each, then EVERY THREAD sorts whole bins of <= 16 entries on its registers (thread_sort16)
//                         and writes them back: the CTA's entry array is then sorted, the rank of position p is
//                         #lower-CTA values + p, and a dense loop emits b = #below, a = #above.  Entries with equal
//                         14-bit keys (true ties, or distinct values closer than 2^-14 of a bin) are compared on the
//                         exact float64 values; bins of 17..255 entries are ranked by a warp by counting.
//
// Exactness: code(x) is non-decreasing in x in exact integer arithmetic (fma is monotone, the table is
// non-decreasing, mulhi is monotone; the two end buckets, which also receive everything outside the range, have
// D = 0), so "lower bin" and "lower key in the same bin" imply a strictly smaller value, and everything else is
// decided on the float64 values themselves.
#pragma once

namespace sd {

constexpr int SL_BUCKETS = 256;        // equal-width buckets; 1 .. SL_BUCKETS-2 cover the row's (trimmed, widened) range
constexpr int SL_SHIFT = 17;           // code = bin << 17 | 17 fractional bits
constexpr int SL_IDBITS = 17;          // entry = key14 << 17 | curve id  (n <= 131072), bit 31 clear
#ifndef SD_SLAB_MEAN
#define SD_SLAB_MEAN 8
#endif
#ifndef SD_SLAB_HIST_MINB
#define SD_SLAB_HIST_MINB 2            // resident hist CTAs per SM the register budget is held to
#endif
constexpr int SL_MEAN = SD_SLAB_MEAN;  // target values per bin
constexpr int SL_SORT_CAP = 16;        // bins of at most this many entries are sorted by one thread
constexpr int SL_BIN_MAX = 255;        // larger bins: the row goes to the generic path
constexpr int SL_TABLE_THREADS = 256;   // table kernel: many small CTAs per SM hide its serial stages
constexpr int SL_HIST_THREADS = 512;    // pass kernel: two CTAs per SM
constexpr int SL_SAMPLE = 16384;       // sampled values per row (quads of 4 consecutive values), 16 per thread
constexpr int SL_SORTED = 1024;        // of which one per thread is sorted for the range
constexpr int SL_DUPS_MAX = 3;         // equal neighbours tolerated in the sorted sample
constexpr int SL_TRIM = 4;             // order statistics of the sorted sample dropped at either end before widening
constexpr i64 SL_MIN_N = SL_SAMPLE;
constexpr i64 SL_MAX_N = 1 << SL_IDBITS;
constexpr u32 SL_PAIRWORK_MAX = 1u << 18;  // sum of cnt^2 over the bins of more than SL_SORT_CAP entries of a row
constexpr u32 SL_IDMASK = (1u << SL_IDBITS) - 1u;
constexpr int SL_TOP0 = 0x43300000;    // high word of 2^52

struct SlabArgs {
    const double *X;
    i64 n, ld;
    int G, NBc, ecap;          // CTAs per row, bins per CTA (a multiple of 1024), entries one CTA may hold
    double2 *rowmap;           // [rows] (s, c): fixed-point position of x = fma(x, s, c)
    uint2 *tables;             // [rows][SL_BUCKETS] (C, D)
    u32 *codes;                // [rows][cpitch] code(x) of every value: written by hist, streamed by the G rank CTAs
    i64 cpitch;                // n rounded up to a multiple of 4
    unsigned short *starts;    // [rows][G*NBc] first entry position of a bin inside its CTA
    u32 *below;                // [rows][G] #values in the bins of lower CTAs
    int *rowflag;              // [rows] 0, or 2: generic path
    int *failcount;            // [0] rows flagged by the table and hist kernels, [1] their CTAs' ticket (slab_report)
    i64 row0;
    int *status;
};

// What the table and hist kernels hand over beside the rows: the unfit-row counts, stored by the last CTA of each kernel
// straight into the host's pinned status mirror (mapped: no copy in the stream between the kernels), and the j = 2
// accumulator of the call, which the table kernel of its first row block clears.
struct SlabReport {
    int *host;                 // device view of the mirror: [0] unfit rows after the hist kernel, [1] after the table kernel
    u64 *zero;                 // [zero_len] cleared by the table kernel, or null
    i64 zero_len;
};

// d = fma(x, s, c) = 2^52 + (1 + (x - lo) * (SL_BUCKETS - 2) / (hi - lo)) * 2^32: the mantissa is a fixed-point
// position, bits 32.. the bucket, bits 0..31 the place inside it.  Values outside the range clamp to the end buckets
// (monotone; their D is 0, so the low word does not matter there).
__device__ __forceinline__ int slab_bucket(const double d) {
    return min(max(__double2hiint(d), SL_TOP0), SL_TOP0 + SL_BUCKETS - 1) - SL_TOP0;
}

// The hist kernel keeps SL_TBL_COPIES copies of the code table, entry k of copy r at word 2 (k * SL_TBL_COPIES + r):
// copy r lies on banks 2r and 2r + 1 whatever k is, so when lane l reads copy l % 16 the lanes of a half-warp hit 16
// different bank pairs and a 64-bit lookup takes its 2 wavefronts for any buckets (one shared table: ~3x that, 71 %
// of the LSU pipe).  tbl points at the lane's copy.
constexpr int SL_TBL_COPIES = 16;

__device__ __forceinline__ u32 slab_code(const double x, const double s, const double c, const uint2 *tbl) {
    const double d = fma(x, s, c);
    const uint2 e = tbl[slab_bucket(d) * SL_TBL_COPIES];
    return e.x + __umulhi((u32)__double2loint(d), e.y);
}

// Thread 0 of every CTA of the table / hist kernel, once its row is decided: the CTA that draws the last ticket stores
// the unfit-row count to the host's mirror; after the hist kernel (always queued behind the table kernel) it also
// resets the count and the ticket, so that every call starts from zeros without a memset.
__device__ __forceinline__ void slab_report(const SlabArgs &a, const SlabReport &r, const bool failed, const bool hist) {
    if (failed) atomicAdd(a.failcount, 1);
    __threadfence();
    if (atomicAdd(a.failcount + 1, 1) != (int)gridDim.x - 1) return;
    __threadfence();
    const int count = hist ? atomicExch(a.failcount, 0) : atomicAdd(a.failcount, 0);
    a.failcount[1] = 0;
    *(volatile int *)(r.host + (hist ? 0 : 1)) = count;
    __threadfence_system();
}

__device__ __forceinline__ bool slab_nonfinite(const double x) {
    return (__double2hiint(x) & 0x7ff00000) == 0x7ff00000;
}

// Streams count vectors through f(vector, index), thread t taking index t, t + nt, ..: four 16-byte loads per thread
// are in flight while the previous four are processed (the consumers are long dependent chains -- fma, table lookup,
// atomic -- so without the double buffer the loads only overlap across warps).
template <class V, class F>
__device__ __forceinline__ void slab_stream(const V *__restrict__ src, const int count, const int tid, const int nt,
                                            F &&f) {
    const int tiles = count / (4 * nt);  // full tiles: every thread has four vectors
    int p0 = tid;
    if (tiles > 0) {
        V v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) v[u] = src[p0 + u * nt];
        for (int t = 1; t <= tiles; ++t) {
            V w[4];
            if (t < tiles) {
#pragma unroll
                for (int u = 0; u < 4; ++u) w[u] = src[p0 + (4 + u) * nt];
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) f(v[u], p0 + u * nt);
            p0 += 4 * nt;
            if (t < tiles) {
#pragma unroll
                for (int u = 0; u < 4; ++u) v[u] = w[u];
            }
        }
    }
    for (; p0 < count; p0 += nt) f(src[p0], p0);
}

// exclusive scan of one value per thread over the CTA (blockDim.x a multiple of 32, <= 1024); wsum: 33 words
__device__ __forceinline__ u32 slab_block_scan(const u32 v, u32 *wsum, u32 &total) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
    u32 incl = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const u32 up = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += up;
    }
    if (lane == 31) wsum[wid] = incl;
    __syncthreads();
    if (wid == 0) {
        const u32 t = lane < nw ? wsum[lane] : 0u;
        u32 sc = t;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const u32 up = __shfl_up_sync(0xffffffffu, sc, d);
            if (lane >= d) sc += up;
        }
        wsum[lane] = sc - t;
        if (lane == 31) wsum[32] = sc;
    }
    __syncthreads();
    total = wsum[32];
    const u32 r = incl - v + wsum[wid];
    __syncthreads();  // wsum may be reused
    return r;
}

// ---------------------------------------------------------------------------------------------
// table: sample -> range and code table.  One small CTA per row (the 55 barrier stages of the sample sort and the
// scattered sample loads are latency, hidden by running many of these CTAs per SM).
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(SL_TABLE_THREADS, 4) mbd_slab_table_kernel(const SlabArgs a, const SlabReport r) {
    __shared__ u32 bh[SL_BUCKETS];
    __shared__ u32 wsum[33];
    __shared__ int s_dups;
    __shared__ float s_q[2];
    const int tid = threadIdx.x;
    const i64 row = blockIdx.x;
    for (i64 i = row * SL_TABLE_THREADS + tid; i < r.zero_len; i += (i64)gridDim.x * SL_TABLE_THREADS) r.zero[i] = 0ull;
    const int n = (int)a.n;
    const double *xr = a.X + row * a.ld;
    const int NB = a.G * a.NBc;
    // The sample: SL_CHUNKS evenly spaced chunks of 256 consecutive values (coalesced 2 KB reads; scattered 32-byte
    // quads cost ~160 bytes of DRAM traffic each, 80 % of a full pass for the whole sample).  Thread t reads value t
    // of every chunk.
    constexpr int SL_CHUNKS = SL_SAMPLE / SL_TABLE_THREADS;  // 64
    const i64 gap = ((i64)n - SL_TABLE_THREADS) / (SL_CHUNKS - 1);  // chunk c starts at c * gap: n >= SL_SAMPLE

    // 1. every 16th value of every chunk (1024 values) is sorted for the range: ONE warp, on its registers, as
    //    order-preserving u32 images of float(x - reference) -- no barrier stages (a 55-stage shared-memory network took
    //    0.09 ms of a 1.2 ms step); the other warps wait
    const double x0 = row_reference(xr, n);
    if (tid < 32) {
        u32 v[32];
        bool bad = false;
#pragma unroll
        for (int i = 0; i < 32; ++i) {
            const int e = tid * 32 + i;
            const double x = xr[(i64)(e >> 4) * gap + ((e & 15) << 4)];
            bad |= slab_nonfinite(x);
            v[i] = f32_sortable(__double2float_rn(x - x0));
        }
        if (bad) atomicOr(a.status, ST_NONFINITE);
        warp_bitonic_sort<32, u32>(v, tid);  // element e = lane * 32 + i, ascending
        int d = 0;
#pragma unroll
        for (int i = 0; i + 1 < 32; ++i) d += v[i] == v[i + 1];
        d += __shfl_down_sync(0xffffffffu, v[0], 1) == v[31] && tid < 31;
#pragma unroll
        for (int k = 16; k > 0; k >>= 1) d += __shfl_xor_sync(0xffffffffu, d, k);
        const u32 klo = __shfl_sync(0xffffffffu, v[SL_TRIM], 0);
        const u32 khi = __shfl_sync(0xffffffffu, v[31 - SL_TRIM], 31);
        if (tid == 0) {
            s_dups = d;
            s_q[0] = f32_unsortable(klo);
            s_q[1] = f32_unsortable(khi);
        }
    }
    bh[tid] = 0u;
    __syncthreads();
    const double qlo = x0 + (double)s_q[0], qhi = x0 + (double)s_q[1];
    const double span = qhi - qlo;
    const double lo = qlo - 0.35 * span, hi = qhi + 0.35 * span;
    const double s = ((double)(SL_BUCKETS - 2) * 4294967296.0) / (hi - lo);
    const double c = (4503599627370496.0 + 4294967296.0) - lo * s;
    // rows with ties (continuous data hardly ever repeats a float image inside a sample of 1024; rounded data does:
    // its equal values would all need the exact path), empty or non-finite ranges: not for this path
    const bool fail = s_dups > SL_DUPS_MAX || !(span > 0.0) || !(s > 0.0) || slab_nonfinite(s) || slab_nonfinite(c);
    if (tid == 0) {
        a.rowflag[row] = fail ? 2 : 0;
        if (!fail) a.rowmap[row] = make_double2(s, c);
        slab_report(a, r, fail, false);
    }
    if (fail) return;  // uniform

    // 2. bucket counts of the whole sample
    for (int c0 = 0; c0 < SL_CHUNKS; c0 += 16) {  // loads do not move across atomics: 16 in flight per round
        double v[16];
#pragma unroll
        for (int u = 0; u < 16; ++u) v[u] = xr[(i64)(c0 + u) * gap + tid];
#pragma unroll
        for (int u = 0; u < 16; ++u) atomicAdd(&bh[slab_bucket(fma(v[u], s, c))], 1u);
    }
    __syncthreads();
    // 3. C[k] = floor(#sample below bucket k * NB * 2^17 / S), D = C[k+1] - C[k]; codes stay below NB << 17 (values
    //    also land in buckets the sample left empty, e.g. beyond its maximum)
    const u32 mine = bh[tid];
    u32 total;
    const u32 excl = slab_block_scan(mine, wsum, total);
    const u32 top = ((u32)NB << SL_SHIFT) - 1u;
    const double scl = (double)top / (double)SL_SAMPLE;
    const u32 c0 = min((u32)((double)excl * scl), top);
    const u32 c1 = min((u32)((double)(excl + mine) * scl), top);
    a.tables[row * SL_BUCKETS + tid] = make_uint2(c0, (tid == 0 || tid == SL_BUCKETS - 1) ? 0u : c1 - c0);
}
static_assert(SL_TABLE_THREADS == SL_BUCKETS && SL_SORTED == 1024 && SL_SORTED == 16 * (SL_SAMPLE / SL_TABLE_THREADS) && SL_TRIM < 32,
              "table kernel layout");

// ---------------------------------------------------------------------------------------------
// hist: ONE pass over the row -> per-value codes, exact bin counts -> starts, validation.  One CTA per row.
// ---------------------------------------------------------------------------------------------
// NT = 512 (two CTAs per SM) when there are rows enough to fill the machine twice over, 1024 (one per SM) for the short
// blocks of a multi-GPU rank or a pipelined host call: a CTA's warps are what hides its DRAM latency.
template <int NT>
__global__ void __launch_bounds__(NT, NT == SL_HIST_THREADS ? SD_SLAB_HIST_MINB : 1)
    mbd_slab_hist_kernel(const SlabArgs a, const SlabReport r) {
    extern __shared__ __align__(16) unsigned char sl_smem[];
    u32 *bins = reinterpret_cast<u32 *>(sl_smem);  // [NB]
    __shared__ uint2 tbl[SL_BUCKETS * SL_TBL_COPIES];  // 32 KB: two CTAs of 512 threads still fit an SM
    __shared__ u32 wsum[33];
    __shared__ u32 s_pairwork;
    __shared__ u32 s_first[32];  // [G] first entry of each rank CTA
    const int tid = threadIdx.x, nt = NT, lane = tid & 31, wid = tid >> 5;
    const i64 row = blockIdx.x;
    if (a.rowflag[row] & 2) {  // the table kernel gave the row up
        if (tid == 0) slab_report(a, r, false, true);
        return;
    }
    const int n = (int)a.n;
    const double *xr = a.X + row * a.ld;
    const int NB = a.G * a.NBc;
    for (int k = tid; k < SL_BUCKETS * SL_TBL_COPIES; k += nt) tbl[k] = a.tables[row * SL_BUCKETS + k / SL_TBL_COPIES];
    for (int b = tid; b < NB; b += nt) bins[b] = 0u;
    if (tid == 0) s_pairwork = 0u;
    const double2 sc = a.rowmap[row];
    const double s = sc.x, c = sc.y;
    const uint2 *tbl_mine = tbl + (lane & (SL_TBL_COPIES - 1));
    __syncthreads();

    // 1. the pass
    bool bad = false;
    u32 *crow = a.codes + row * a.cpitch;
    uint2 *crow2 = reinterpret_cast<uint2 *>(crow);
    slab_stream(reinterpret_cast<const double2 *>(xr), n >> 1, tid, nt, [&](const double2 v, const int p) {
        bad |= slab_nonfinite(v.x) | slab_nonfinite(v.y);
        const u32 c0 = slab_code(v.x, s, c, tbl_mine), c1 = slab_code(v.y, s, c, tbl_mine);
        crow2[p] = make_uint2(c0, c1);
        atomicAdd(&bins[c0 >> SL_SHIFT], 1u);
        atomicAdd(&bins[c1 >> SL_SHIFT], 1u);
    });
    if ((n & 1) && tid == 0) {
        bad |= slab_nonfinite(xr[n - 1]);
        const u32 c0 = slab_code(xr[n - 1], s, c, tbl_mine);
        crow[n - 1] = c0;
        atomicAdd(&bins[c0 >> SL_SHIFT], 1u);
    }
    if (bad) atomicOr(a.status, ST_NONFINITE);
    __syncthreads();

    // 2. exclusive prefix over the bins (in place), validation, per-CTA starts.  Warp w owns the bins
    //    [w * S, (w + 1) * S) (S a multiple of 32: NB is a multiple of 1024) and its lanes walk them 32 consecutive
    //    bins at a time, so that every shared-memory access is conflict-free; a warp scan carries the running sum.
    const int S = NB / (NT / 32);
    u32 *wbins = bins + wid * S + lane;
    u32 sum = 0u, maxc = 0u, pairwork = 0u;
    for (int k = 0; k < S; k += 32) {
        const u32 cnt = wbins[k];
        sum += cnt;
        maxc = max(maxc, cnt);
        if (cnt > (u32)SL_SORT_CAP) pairwork += min(cnt, 65535u) * min(cnt, 65535u);
    }
    if (pairwork) atomicAdd(&s_pairwork, min(pairwork, SL_PAIRWORK_MAX + 1u));
    u32 total;
    u32 run = __shfl_sync(0xffffffffu, slab_block_scan(sum, wsum, total), 0);  // values in lower warps' bins
    for (int k = 0; k < S; k += 32) {
        const u32 cnt = wbins[k];
        u32 incl = cnt;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const u32 up = __shfl_up_sync(0xffffffffu, incl, d);
            if (lane >= d) incl += up;
        }
        wbins[k] = run + incl - cnt;
        run += __shfl_sync(0xffffffffu, incl, 31);
    }
    __syncthreads();
    bool fail = maxc > (u32)SL_BIN_MAX || total != (u32)n;
    if (tid < a.G) {
        const u32 first = bins[tid * a.NBc];
        const u32 next = tid + 1 < a.G ? bins[(tid + 1) * a.NBc] : (u32)n;
        fail |= next - first > (u32)a.ecap;
        a.below[row * a.G + tid] = first;
        s_first[tid] = first;
    }
    if (tid == 0) fail |= s_pairwork > SL_PAIRWORK_MAX;
    fail = __syncthreads_or(fail);
    if (tid == 0) slab_report(a, r, fail, true);
    if (fail) {
        if (tid == 0) a.rowflag[row] = 2;
        return;
    }
    // starts relative to the owning rank CTA's first bin, copied out coalesced (two per word; NBc is even, so both
    // bins of a word belong to the same rank CTA)
    const uint2 *bins2 = reinterpret_cast<const uint2 *>(bins);
    u32 *st2 = reinterpret_cast<u32 *>(a.starts + row * NB);  // NB is a multiple of 1024
    const int words_c = a.NBc >> 1;
    int g = 0, edge = words_c;  // rank CTA of word w, first word of the next one
    for (int w = tid; w < (NB >> 1); w += nt) {
        while (w >= edge) {
            ++g;
            edge += words_c;
        }
        const uint2 v = bins2[w];
        const u32 first = s_first[g];
        st2[w] = (v.x - first) | ((v.y - first) << 16);
    }
}

// ---------------------------------------------------------------------------------------------
// rank: grid (G, rows); CTA g of a row keeps and ranks the values of bins [g*NBc, (g+1)*NBc)
// ---------------------------------------------------------------------------------------------
// exact rank of entry m of bin [start, start + cnt): keys first, float64 values where the keys are equal
template <bool EXTRA>
__device__ __noinline__ void slab_rank_entry(const u32 *ents, const int start, const int cnt, const int m,
                                             const double *__restrict__ xr, const u32 before, const RankOut &o,
                                             const i64 row_global, const i64 acc_off) {
    const u32 mine = ents[start + m];
    const u32 km = mine >> SL_IDBITS;
    u32 less = 0u, eq = 1u;
    for (int f = 0; f < cnt; ++f) {
        const u32 other = ents[start + f];
        const u32 ko = other >> SL_IDBITS;
        less += ko < km;
        if (ko == km && f != m) {
            const double xo = xr[other & SL_IDMASK], xm = xr[mine & SL_IDMASK];
            less += xo < xm;
            eq += xo == xm;
        }
    }
    const u32 b = before + less;
    emit_rank<EXTRA>(o, row_global, acc_off, mine & SL_IDMASK, b, (u32)o.n - b - eq);
}

// keeps a value (its code, its curve id) if its bin belongs to this CTA: one atomic on the bin's running position
// places the entry.  word_sa / ents_sa: 32-bit shared-window addresses (the generic-pointer form re-derives the
// window base for every store: four uniform-datapath instructions per value).
__device__ __forceinline__ void slab_keep(const u32 code, const u32 id, const u32 word_sa, const u32 ents_sa,
                                          const u32 base_bin, const u32 NBc) {
    const u32 own = (code >> SL_SHIFT) - base_bin;
    if (own < NBc) {
        u32 pos;
        asm volatile("atom.shared.add.u32 %0, [%1], 1;" : "=r"(pos) : "r"(word_sa + 4u * own) : "memory");
        asm volatile("st.shared.u32 [%0], %1;" ::"r"(ents_sa + 4u * pos), "r"(((code << 14) & 0x7ffe0000u) | id)
                     : "memory");
    }
}

template <bool EXTRA>
__global__ void __launch_bounds__(1024, 1) mbd_slab_rank_kernel(const SlabArgs a, const RankOut o) {
    extern __shared__ __align__(16) unsigned char sl_smem[];
    u32 *ents = reinterpret_cast<u32 *>(sl_smem);                        // [ecap + SL_SORT_CAP]
    u32 *word = ents + a.ecap + SL_SORT_CAP;                             // [NBc] running position: start, then end
    const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, wid = tid >> 5, nw = nt >> 5;
    const i64 row = blockIdx.y;
    const int g = blockIdx.x;
    if (a.rowflag[row] & 2) return;  // the whole row goes to the generic path
    const int n = (int)a.n;
    const int NBc = a.NBc;
    const double *xr = a.X + row * a.ld;
    {
        const unsigned short *st = a.starts + (row * a.G + g) * NBc;
        for (int b = tid; b < NBc; b += nt) word[b] = st[b];
    }
    const u32 bel = a.below[row * a.G + g];
    const u32 base_bin = (u32)g * (u32)NBc;
    __syncthreads();

    // 1. stream the row's codes; keep the values of this CTA's bins
    {
        const u32 nbc = (u32)NBc;
        const u32 ents_sa = (u32)__cvta_generic_to_shared(ents), word_sa = (u32)__cvta_generic_to_shared(word);
        const u32 *crow = a.codes + row * a.cpitch;
        slab_stream(reinterpret_cast<const uint4 *>(crow), n >> 2, tid, nt, [&](const uint4 v, const int p) {
            const u32 id = 4u * (u32)p;
            slab_keep(v.x, id, word_sa, ents_sa, base_bin, nbc);
            slab_keep(v.y, id + 1u, word_sa, ents_sa, base_bin, nbc);
            slab_keep(v.z, id + 2u, word_sa, ents_sa, base_bin, nbc);
            slab_keep(v.w, id + 3u, word_sa, ents_sa, base_bin, nbc);
        });
        const int c = (n & ~3) + tid;
        if (c < n) slab_keep(crow[c], (u32)c, word_sa, ents_sa, base_bin, nbc);
    }
    __syncthreads();

    // 2. every thread sorts whole bins on its registers and emits their ranks: entry i of the sorted bin has
    //    bel + start + i values below it.  word[b] is now the END of bin b (= the start of bin b + 1).  Lane l owns the
    //    stripe [l*Qs, (l+1)*Qs) of the CTA's bins and walks it rotated by l, so that the lanes' words fall into
    //    different banks; every warp does exactly Qs / nw rounds.  The scattered 8-byte REDs of the emission (one L2
    //    request each) overlap with the next bin's sort.  A bin of more than 16 entries, or one with equal keys
    //    (0.5 % of the bins), is ranked by the whole warp on the exact values right away.
    const i64 row_global = a.row0 + row;
    const i64 acc_off = EXTRA ? acc_offset(o, row_global) : 0;
    const u32 n1 = (u32)n - 1u;
    const int Qs = NBc >> 5;
    for (int q = wid; q < Qs; q += nw) {  // warp-uniform trip count
        int t = q + lane;
        if (t >= Qs) t -= Qs;
        const int b = lane * Qs + t;
        const int start = b > 0 ? (int)word[b - 1] : 0;
        const int cnt = (int)word[b] - start;
        u32 e[SL_SORT_CAP];  // pads: above every entry (bit 31), 2^20 apart
#pragma unroll
        for (int i = 0; i < SL_SORT_CAP; ++i) {
            const u32 v = ents[start + i];
            e[i] = i < cnt ? v : 0x80000000u + ((u32)i << 20);
        }
        thread_sort16<u32>(e);
        // neighbours closer than 2^17 may share their key (conservative: a key step with descending ids also counts)
        u32 gap = 0xffffffffu;
#pragma unroll
        for (int i = 0; i + 1 < SL_SORT_CAP; ++i) gap = min(gap, e[i + 1] - e[i]);
        const bool plain = cnt <= SL_SORT_CAP && gap >= (1u << SL_IDBITS);
        if (plain) {
            const u32 before = bel + (u32)start;
            if (EXTRA) {  // rank output / j = 3 / row groups: a rolled loop over the written-back bin (registers)
#pragma unroll
                for (int i = 0; i < SL_SORT_CAP; ++i)
                    if (i < cnt) ents[start + i] = e[i];
#pragma unroll 1
                for (int i = 0; i < cnt; ++i)
                    emit_rank<EXTRA>(o, row_global, acc_off, ents[start + i] & SL_IDMASK, before + i, n1 - before - i);
            } else {
#pragma unroll
                for (int i = 0; i < SL_SORT_CAP; ++i)
                    if (i < cnt) emit_rank<EXTRA>(o, row_global, acc_off, e[i] & SL_IDMASK, before + i, n1 - before - i);
            }
        }
        unsigned todo = __ballot_sync(0xffffffffu, !plain);
        while (todo) {  // rare
            const int src = __ffs(todo) - 1;
            todo &= todo - 1;
            const int bs = __shfl_sync(0xffffffffu, start, src), bc = __shfl_sync(0xffffffffu, cnt, src);
            for (int m = lane; m < bc; m += 32)
                slab_rank_entry<EXTRA>(ents, bs, bc, m, xr, bel + (u32)bs, o, row_global, acc_off);
        }
    }
}

}  // namespace sd
