// bd_match.cu -- strict band depth (J = 2) by matching complementary sign vectors: O(nT) per query.
//
// Same quantity as bd_bits.cu / bd_gemm.cu (strict branch of _r2_containment, _containment.py:68-80,
// over all pairs, _functional.py:238-253), different algorithm.  For query q let B_o / A_o be the T-bit
// vectors "other curve o is strictly below / above q".  A pair (o1, o2) contains q at every time point
// iff B_o1 & B_o2 == 0 and A_o1 & A_o2 == 0.  If neither curve ever ties with q (A = ~B), that is
// EXACTLY  B_o2 == A_o1: the two sign vectors are complements.  So for the tie-free curves F
//     #pairs in F x F  =  1/2 * sum_{o in F} #{o' in F : B_o' == A_o}
// which is a dictionary lookup, not a pair enumeration:
//   bd_sig_rank_kernel : sign words (one fixed bit order), a 64-bit hash of B_o and of its complement, and a
//                     tie-free flag per (query, other curve); 8 queries per thread.  Works on the per-time-point
//                     RANKS of the curves (one pass of the mbd.cu rank pipeline), two 15-bit compares per
//                     32-bit subtraction.  bd_sig_kernel is the float64 variant for few queries / long series.
//   bd_match_kernel : one CTA per query sorts the (hash | curve id) keys of the tie-free curves (register
//                     bitonic network on u64 + swizzled shared-memory merges), checks that every run of
//                     equal hashes holds ONE sign vector (word-by-word), looks every curve's complement up by
//                     binary search, confirms the match word-by-word and adds the run length.  The few
//                     curves that tie with q somewhere (set Z, at most 64) are tested against everybody.
// Exactness does not rest on the hash: a run with two different vectors, a hash hit whose words differ, or
// more than 64 tied curves flags the query, and flagged queries are recomputed by the enumerating kernels.
// Both drivers, for one matrix and for nb equally shaped matrices (permutation tests), take their ranks from
// packed_ranks (one rank pass, ranks packed in pairs; the single driver skips it for long series or few queries)
// and end in recompute_flagged (flags read back once, flagged queries recomputed matrix by matrix).  They differ
// in how they chunk the signature and match launches.
#include <vector>

#include "common.cuh"
#include "sortnet.cuh"

namespace sd {

constexpr int BM_SQ = 8;           // queries per thread in the signature kernel
constexpr int BM_THREADS = 512;    // match kernel: 16 warps x 512 keys
constexpr int BM_EPL = 16;
constexpr int BM_MAXM = 8192;      // sort capacity = most other curves per query
constexpr int BM_ZCAP = 64;
constexpr u64 BM_IDMASK = 0x1fffull;  // low 13 bits carry the curve position

__device__ __forceinline__ u64 bm_mix(u64 h, u32 w) {
    h ^= (u64)w;
    h *= 0x9E3779B97F4A7C15ull;
    h ^= h >> 29;
    return h;
}
__device__ __forceinline__ u64 bm_final(u64 h) {
    h ^= h >> 32;
    h *= 0xD6E8FEB86659FD93ull;
    h ^= h >> 32;
    return h;
}

// Mw[(q*W + w)*m + o] = {below, above} bits of time points 32w .. 32w+31 (first time point in the highest used bit);
// sig[q*m + o] = {hash(B), hash(~B & valid)};  tf[q*m + o] = 1 iff o never ties with q.
__global__ void __launch_bounds__(128) bd_sig_kernel(const double *__restrict__ X, const i64 T, const i64 n,
                                                     const i64 ld, const i64 *__restrict__ qidx, const int nqb,
                                                     const int W, uint2 *__restrict__ Mw, ulonglong2 *__restrict__ sig,
                                                     unsigned char *__restrict__ tf, int *__restrict__ status) {
    __shared__ double sq[32][BM_SQ];
    __shared__ i64 sqi[BM_SQ];
    const int q0 = blockIdx.y * BM_SQ;
    if (threadIdx.x < BM_SQ) sqi[threadIdx.x] = q0 + threadIdx.x < nqb ? qidx[q0 + threadIdx.x] : -1;
    const i64 m = n - 1;
    // one thread per CURVE c; for query q it is other curve o = c - [c > q] (and nothing when c == q)
    const i64 c = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = c < n;
    u64 hb[BM_SQ], hc[BM_SQ];
    bool tiefree[BM_SQ];
#pragma unroll
    for (int qq = 0; qq < BM_SQ; ++qq) {
        hb[qq] = hc[qq] = 0x243F6A8885A308D3ull;
        tiefree[qq] = true;
    }
    bool bad = false;
    for (int w = 0; w < W; ++w) {
        __syncthreads();
        for (int i = threadIdx.x; i < 32 * BM_SQ; i += blockDim.x) {
            const int tt = i / BM_SQ, qq = i % BM_SQ;
            const i64 t = (i64)w * 32 + tt;
            sq[tt][qq] = (t < T && sqi[qq] >= 0) ? X[t * ld + sqi[qq]] : 0.0;
        }
        __syncthreads();
        if (!live) continue;
        const int tmax = (T - (i64)w * 32) < 32 ? (int)(T - (i64)w * 32) : 32;
        const u32 valid = tmax == 32 ? 0xffffffffu : ((1u << tmax) - 1u);
        u32 b[BM_SQ], a[BM_SQ];
#pragma unroll
        for (int qq = 0; qq < BM_SQ; ++qq) b[qq] = a[qq] = 0u;
        const double *col = X + (i64)w * 32 * ld + c;
#pragma unroll 8
        for (int tt = 0; tt < tmax; ++tt) {
            const double x = col[(i64)tt * ld];
            bad |= !isfinite(x);
#pragma unroll
            for (int qq = 0; qq < BM_SQ; ++qq) {
                // shift-in as 2*w + bit: a multiply-add (FMA pipe) instead of shift + or on the ALU pipe, which
                // this kernel keeps 78 % busy.  Time point tt lands in bit tmax-1-tt of the word: any fixed bit
                // order serves (words are only compared with, and ANDed against, words built the same way).
                const double xq = sq[tt][qq];
                b[qq] = b[qq] * 2u + (u32)(x < xq);
                a[qq] = a[qq] * 2u + (u32)(x > xq);
            }
        }
#pragma unroll
        for (int qq = 0; qq < BM_SQ; ++qq) {
            const i64 qi = sqi[qq];
            if (qi >= 0 && c != qi) Mw[((i64)(q0 + qq) * W + w) * m + (c - (c > qi))] = make_uint2(b[qq], a[qq]);
            hb[qq] = bm_mix(hb[qq], b[qq]);
            hc[qq] = bm_mix(hc[qq], ~b[qq] & valid);
            tiefree[qq] = tiefree[qq] && ((b[qq] | a[qq]) == valid);
        }
    }
    if (bad) atomicOr(status, ST_NONFINITE);
    if (!live) return;
#pragma unroll
    for (int qq = 0; qq < BM_SQ; ++qq) {
        const i64 qi = sqi[qq];
        if (qi >= 0 && c != qi) {
            const i64 o = c - (c > qi);
            sig[(i64)(q0 + qq) * m + o] = make_ulonglong2(bm_final(hb[qq]), bm_final(hc[qq]));
            tf[(i64)(q0 + qq) * m + o] = tiefree[qq] ? 1 : 0;
        }
    }
}


// ---------------------------------------------------------------------------------------------
// Signatures from RANKS.  At one time point "x_o < x_q" is "rank_o < rank_q" when rank = number of curves
// strictly below (ties share a rank), so the per-row rank pipeline of mbd.cu turns the float64 compares of
// every (query, curve, time point) into 15-bit integer compares, two per 32-bit subtraction:
//     d = (r2 | 0x80008000) - q2  has bit 15 / 31 set  iff  r >= q  in the low / high half (no borrow between the
// halves), and d - 0x00010001 has them set iff r > q.  ~3 warp instructions per 32 comparisons instead of ~11
// with DSETP + predicate-to-bit.
// Word layout (any fixed order serves): bit k <-> time point 32w + 2k, bit 16 + k <-> time point 32w + 2k + 1.
// ---------------------------------------------------------------------------------------------
constexpr u32 BM_GUARD = 0x80008000u;

// Rp[tp*n + c] = rank[2tp][c] | rank[2tp+1][c] << 16; time points past T get rank 0 for everybody (a tie)
// (blockIdx.y = batch: every batch has its own T rank rows and TP packed rows)
__global__ void bd_pack_ranks_kernel(const int *__restrict__ rank_b, const i64 T, const i64 n, const i64 TP,
                                     u32 *__restrict__ Rp) {
    rank_b += (i64)blockIdx.y * T * n;
    Rp += (i64)blockIdx.y * TP * n;
    const i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= TP * n) return;
    const i64 tp = i / n, c = i - tp * n;
    const i64 t0 = 2 * tp, t1 = t0 + 1;
    const u32 lo = t0 < T ? (u32)rank_b[t0 * n + c] : 0u;
    const u32 hi = t1 < T ? (u32)rank_b[t1 * n + c] : 0u;
    Rp[i] = lo | (hi << 16);
}

// blockIdx.z = batch (batched permutation calls): every batch has its own packed ranks, nqb queries and outputs
__global__ void __launch_bounds__(128) bd_sig_rank_kernel(const u32 *__restrict__ Rp, const i64 T, const i64 n,
                                                          const i64 *__restrict__ qidx, const int nqb, const int W,
                                                          uint2 *__restrict__ Mw, ulonglong2 *__restrict__ sig,
                                                          unsigned char *__restrict__ tf) {
    __shared__ u32 sq[16][BM_SQ];
    __shared__ i64 sqi[BM_SQ];
    {
        const i64 z = blockIdx.z;
        Rp += z * (i64)W * 16 * n;
        qidx += z * nqb;
        Mw += z * (i64)nqb * W * (n - 1);
        sig += z * (i64)nqb * (n - 1);
        tf += z * (i64)nqb * (n - 1);
    }
    const int q0 = blockIdx.y * BM_SQ;
    if (threadIdx.x < BM_SQ) sqi[threadIdx.x] = q0 + threadIdx.x < nqb ? qidx[q0 + threadIdx.x] : -1;
    const i64 m = n - 1;
    const i64 c = (i64)blockIdx.x * blockDim.x + threadIdx.x;  // one thread per CURVE, BM_SQ queries each
    const bool live = c < n;
    u64 hb[BM_SQ], hc[BM_SQ];
    bool tiefree[BM_SQ];
#pragma unroll
    for (int qq = 0; qq < BM_SQ; ++qq) {
        hb[qq] = hc[qq] = 0x243F6A8885A308D3ull;
        tiefree[qq] = true;
    }
    for (int w = 0; w < W; ++w) {
        __syncthreads();
        for (int i = threadIdx.x; i < 16 * BM_SQ; i += blockDim.x) {
            const int k = i / BM_SQ, qq = i % BM_SQ;
            sq[k][qq] = sqi[qq] >= 0 ? Rp[((i64)w * 16 + k) * n + sqi[qq]] : 0u;
        }
        __syncthreads();
        if (!live) continue;
        const i64 rem = T - (i64)w * 32;  // >= 1
        const int n_even = rem >= 31 ? 16 : (int)((rem + 1) >> 1), n_odd = rem >= 32 ? 16 : (int)(rem >> 1);
        const u32 valid = ((1u << n_even) - 1u) | (((1u << n_odd) - 1u) << 16);
        const u32 *col = Rp + (i64)w * 16 * n + c;
        u32 r2[16];
#pragma unroll
        for (int k = 0; k < 16; ++k) r2[k] = col[(i64)k * n];
        u32 ge[BM_SQ], gt[BM_SQ];
#pragma unroll
        for (int qq = 0; qq < BM_SQ; ++qq) ge[qq] = gt[qq] = 0u;
#pragma unroll
        for (int k = 0; k < 16; ++k) {
            const u32 rg = r2[k] | BM_GUARD;
#pragma unroll
            for (int qq = 0; qq < BM_SQ; ++qq) {
                // d = rg - q2: guard bits = [r >= q];  d - 0x00010001: guard bits = [r >= q + 1] = [r > q] (each
                // half of d is >= 1, so neither subtraction borrows across the halves).  Both differences are
                // written as multiply-adds: the kernel is bound by the ALU pipe, the FMA pipe is idle.
                const u32 q2 = sq[k][qq];
                u32 d, d1;
                asm("mad.lo.u32 %0, %1, 0xffffffff, %2;" : "=r"(d) : "r"(q2), "r"(rg));
                asm("mad.lo.u32 %0, %1, 1, 0xfffeffff;" : "=r"(d1) : "r"(d));
                ge[qq] = (ge[qq] >> 1) | (d & BM_GUARD);
                gt[qq] = (gt[qq] >> 1) | (d1 & BM_GUARD);
            }
        }
#pragma unroll
        for (int qq = 0; qq < BM_SQ; ++qq) {
            const u32 b = ~ge[qq] & valid, a = gt[qq] & valid;
            const i64 qi = sqi[qq];
            if (qi >= 0 && c != qi) Mw[((i64)(q0 + qq) * W + w) * m + (c - (c > qi))] = make_uint2(b, a);
            hb[qq] = bm_mix(hb[qq], b);
            hc[qq] = bm_mix(hc[qq], ~b & valid);
            tiefree[qq] = tiefree[qq] && ((b | a) == valid);
        }
    }
    if (!live) return;
#pragma unroll
    for (int qq = 0; qq < BM_SQ; ++qq) {
        const i64 qi = sqi[qq];
        if (qi >= 0 && c != qi) {
            const i64 o = c - (c > qi);
            sig[(i64)(q0 + qq) * m + o] = make_ulonglong2(bm_final(hb[qq]), bm_final(hc[qq]));
            tf[(i64)(q0 + qq) * m + o] = tiefree[qq] ? 1 : 0;
        }
    }
}

__device__ __forceinline__ int bm_swz(int g) { return g ^ ((g >> 4) & 15); }

// 51-bit hash field of a key; the all-ones value is reserved for the sentinel (sorts last)
__device__ __forceinline__ u64 bm_h51(u64 h) {
    const u64 x = h >> 13;
    return x == 0x7ffffffffffffull ? x - 1 : x;
}

// B words of curve o equal the B words of curve p?
__device__ __forceinline__ bool bm_same_b(const uint2 *__restrict__ Mq, const int W, const i64 m, const int o,
                                          const int p) {
    for (int w = 0; w < W; ++w)
        if (Mq[(i64)w * m + o].x != Mq[(i64)w * m + p].x) return false;
    return true;
}
// complement of o's B words equals p's B words?  o is tie-free, so its A words ARE that complement (within the
// valid bits, whatever the bit order of the words).
__device__ __forceinline__ bool bm_complement(const uint2 *__restrict__ Mq, const int W, const i64 m, const int o,
                                              const int p) {
    for (int w = 0; w < W; ++w)
        if (Mq[(i64)w * m + o].y != Mq[(i64)w * m + p].x) return false;
    return true;
}

// one CTA per query; flag[q] = 1 asks the caller to recompute the query with an enumerating kernel
// NT threads sort up to 16 * NT keys: NT = 512 for the general case (m <= 8192), NT = 64 / 32 when the other
// curves of a query fit 1024 / 512 keys (permutation batches), where a 8192-slot sort would be 16-32x overwork.
template <int NT>
__global__ void __launch_bounds__(NT, NT == 512 ? 2 : 8) bd_match_kernel(const uint2 *__restrict__ Mw,
                                                              const ulonglong2 *__restrict__ sig,
                                                              const unsigned char *__restrict__ tf, const i64 m,
                                                              const i64 T, const int W, i64 *__restrict__ out,
                                                              unsigned char *__restrict__ flag) {
    extern __shared__ __align__(16) unsigned char bm_smem[];
    u64 *skey = reinterpret_cast<u64 *>(bm_smem);  // (NT * 16) keys
    {   // blockIdx.y = batch: gridDim.x queries per batch
        const i64 z = (i64)blockIdx.y * gridDim.x;
        Mw += z * W * m;
        sig += z * m;
        tf += z * m;
        out += z;
        flag += z;
    }
    __shared__ int s_z[BM_ZCAP];
    __shared__ int s_nz, s_bad;
    __shared__ u64 s_red[NT / 32];
    const int q = blockIdx.x;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const uint2 *Mq = Mw + (i64)q * W * m;
    const ulonglong2 *sg = sig + (i64)q * m;
    const unsigned char *tq = tf + (i64)q * m;
    if (tid == 0) { s_nz = 0; s_bad = 0; }
    __syncthreads();

    // 1. keys of the tie-free curves (hash in the high 51 bits, position in the low 13); the rest is Z
    u64 v[BM_EPL];
#pragma unroll
    for (int i = 0; i < BM_EPL; ++i) {
        const int o = wid * 512 + lane * BM_EPL + i;
        u64 key = ~0ull;
        if (o < m) {
            if (tq[o]) {
                key = (bm_h51(sg[o].x) << 13) | (u64)o;
            } else {
                const int z = atomicAdd(&s_nz, 1);
                if (z < BM_ZCAP) s_z[z] = o;
            }
        }
        v[i] = key;
    }
    // 2. sort: 512 keys per warp on registers, then 4 merge levels through swizzled shared memory
    warp_bitonic_sort<BM_EPL, u64>(v, lane);
    for (int k = 1024; k <= (NT * 16); k <<= 1) {
        for (int j = k; j >= 1024; j >>= 1) {  // j == k: mirror stage (g ^ (k-1)); else xor stage (g ^ j/2)
            __syncthreads();
#pragma unroll
            for (int i = 0; i < BM_EPL; ++i) skey[bm_swz(wid * 512 + lane * BM_EPL + i)] = v[i];
            __syncthreads();
            const int xorv = (j == k) ? (k - 1) : (j >> 1);
            const bool lower = ((wid * 512) & (j == k ? (k >> 1) : (j >> 1))) == 0;
#pragma unroll
            for (int i = 0; i < BM_EPL; ++i) {
                const u64 o = skey[bm_swz((wid * 512 + lane * BM_EPL + i) ^ xorv)];
                v[i] = lower ? min(v[i], o) : max(v[i], o);
            }
        }
        warp_merge_tail<BM_EPL, u64>(v, lane, 16);  // strides 256 .. 1 stay inside the warp
    }
    __syncthreads();
#pragma unroll
    for (int i = 0; i < BM_EPL; ++i) skey[bm_swz(wid * 512 + lane * BM_EPL + i)] = v[i];
    __syncthreads();
    const int nz_all = s_nz;
    const int nz = nz_all < BM_ZCAP ? nz_all : BM_ZCAP;
    const int nF = (int)m - nz_all;  // tie-free keys occupy sorted positions [0, nF)
    bool bad = nz_all > BM_ZCAP;

    // 3. every run of equal hashes must hold one sign vector; look up every curve's complement
    u64 twice = 0;  // sum over o in F of #{o' in F : B_o' == A_o}
    for (int p = tid; p < nF && !bad; p += NT) {
        const u64 key = skey[bm_swz(p)];
        const int o = (int)(key & BM_IDMASK);
        const u64 h = key >> 13;
        if (p > 0) {
            const u64 prev = skey[bm_swz(p - 1)];
            if ((prev >> 13) == h && !bm_same_b(Mq, W, m, o, (int)(prev & BM_IDMASK))) bad = true;
        }
        const u64 target = bm_h51(sg[o].y);
        int lo = 0, hi = nF;  // first position with hash >= target
        while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if ((skey[bm_swz(mid)] >> 13) < target) lo = mid + 1; else hi = mid;
        }
        if (lo < nF && (skey[bm_swz(lo)] >> 13) == target) {
            const int rep = (int)(skey[bm_swz(lo)] & BM_IDMASK);
            if (bm_complement(Mq, W, m, o, rep)) {
                int l2 = lo, h2 = nF;  // first position with hash > target
                while (l2 < h2) {
                    const int mid = (l2 + h2) >> 1;
                    if ((skey[bm_swz(mid)] >> 13) <= target) l2 = mid + 1; else h2 = mid;
                }
                twice += (u64)(l2 - lo);
            } else {
                bad = true;  // hash hit with different words: let the enumerating kernel decide
            }
        }
    }
    // 4. curves that tie with the query somewhere: test them against everybody (pairs inside Z once)
    u64 zc = 0;
    if (!bad) {
        for (int zi = 0; zi < nz; ++zi) {
            const int z = s_z[zi];
            for (int o = tid; o < m; o += NT) {
                if (o == z || (!tq[o] && o < z)) continue;
                bool ok = true;
                for (int w = 0; w < W && ok; ++w) {
                    const uint2 a = Mq[(i64)w * m + z], b = Mq[(i64)w * m + o];
                    ok = ((a.x & b.x) | (a.y & b.y)) == 0u;
                }
                zc += ok;
            }
        }
    }
    if (bad) atomicOr(&s_bad, 1);
    u64 tot = twice + 2 * zc;  // halve at the end (twice is even)
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) tot += __shfl_xor_sync(0xffffffffu, tot, s);
    if (lane == 0) s_red[wid] = tot;
    __syncthreads();
    if (tid == 0) {
        u64 t2 = 0;
        for (int w = 0; w < NT / 32; ++w) t2 += s_red[w];
        out[q] = (i64)(t2 >> 1);
        flag[q] = s_bad ? 1 : 0;
    }
}

__global__ void bm_scatter_kernel(const i64 *__restrict__ src, const i64 *__restrict__ pos, i64 cnt,
                                  i64 *__restrict__ dst) {
    const i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < cnt) dst[pos[i]] = src[i];
}

// picks the smallest sort capacity that holds the m other curves of a query
static int launch_match(cudaStream_t st, dim3 grid, i64 m, const uint2 *Mw, const ulonglong2 *sig,
                        const unsigned char *tf, i64 T, int W, i64 *out, unsigned char *flag) {
    if (m <= 512) {
        bd_match_kernel<32><<<grid, 32, 32 * 16 * sizeof(u64), st>>>(Mw, sig, tf, m, T, W, out, flag);
    } else if (m <= 1024) {
        bd_match_kernel<64><<<grid, 64, 64 * 16 * sizeof(u64), st>>>(Mw, sig, tf, m, T, W, out, flag);
    } else {
        const size_t smem = (size_t)BM_MAXM * sizeof(u64);
        SD_CUDA(cudaFuncSetAttribute(bd_match_kernel<BM_THREADS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        bd_match_kernel<BM_THREADS><<<grid, BM_THREADS, smem, st>>>(Mw, sig, tf, m, T, W, out, flag);
    }
    SD_CUDA(cudaGetLastError());
    return SD_OK;
}

bool bd_match_supported(i64 T, i64 n) { return n - 1 <= BM_MAXM && n >= 3 && ceil_div(T, 32) <= 4096; }

// Ranks of all curves at every time point of nb matrices of T rows (matrix b starts at row b·T of dX), from one pass
// of the rank pipeline, packed in pairs for the signature kernel: *Rp = [nb][TP][n] words in BUF_RANKS.
static int packed_ranks(sd_ctx *ctx, const double *dX, i64 ld, i64 nb, i64 T, i64 n, u32 **Rp) {
    const i64 TP = ceil_div(T, 32) * 16;
    SD_TRY(ctx->buf[BUF_RANKS].reserve((size_t)nb * T * n * sizeof(int) + (size_t)nb * TP * n * sizeof(u32)));
    int *rank_b = ctx->buf[BUF_RANKS].as<int>();
    *Rp = reinterpret_cast<u32 *>(rank_b + (size_t)nb * T * n);
    SD_TRY(rank_rows_device(ctx, dX, nb * T, n, ld, rank_b, nullptr));
    SD_TRY(prof_begin(ctx, SD_PHASE_BD_MASKS));
    for (i64 b0 = 0; b0 < nb; b0 += 65535) {  // gridDim.y = batch: at most 65 535 per launch
        const i64 cb = nb - b0 < 65535 ? nb - b0 : 65535;
        bd_pack_ranks_kernel<<<dim3((unsigned)ceil_div(TP * n, 256), (unsigned)cb), 256, 0, ctx->stream>>>(
            rank_b + b0 * T * n, T, n, TP, *Rp + b0 * TP * n);
        ctx->last.launches++;
    }
    SD_TRY(prof_end(ctx));
    return SD_OK;
}

// Recomputes the queries the match kernel flagged with `fallback` (the enumerating path), matrix by matrix: nb
// matrices of T rows (matrix b starts at row b·T of dX), nqb queries each, d_flag / d_q / d_out laid out [nb][nqb].
// Reads the flags back with one synchronisation; *n_fallback (if given) grows by the number of flagged queries.
static int recompute_flagged(sd_ctx *ctx, const double *dX, i64 nb, i64 T, i64 n, i64 ld, const i64 *d_q, i64 nqb,
                             const unsigned char *d_flag, i64 *d_out, StrictFallback fallback, i64 *n_fallback) {
    cudaStream_t st = ctx->stream;
    std::vector<unsigned char> h_flag((size_t)(nb * nqb));
    SD_CUDA(cudaMemcpyAsync(h_flag.data(), d_flag, h_flag.size(), cudaMemcpyDeviceToHost, st));
    SD_CUDA(cudaStreamSynchronize(st));
    std::vector<i64> pos;
    for (i64 b = 0; b < nb; ++b) {
        pos.clear();
        for (i64 i = 0; i < nqb; ++i)
            if (h_flag[(size_t)(b * nqb + i)]) pos.push_back(i);
        if (n_fallback) *n_fallback += (i64)pos.size();
        if (pos.empty()) continue;
        const i64 nf = (i64)pos.size();
        SD_TRY(ctx->buf[BUF_SPLIT].reserve((size_t)nf * 3 * sizeof(i64)));
        i64 *d_pos = ctx->buf[BUF_SPLIT].as<i64>();
        i64 *d_qsub = d_pos + nf, *d_osub = d_qsub + nf;
        SD_CUDA(cudaMemcpyAsync(d_pos, pos.data(), (size_t)nf * sizeof(i64), cudaMemcpyHostToDevice, st));
        SD_TRY(gather_i64_device(ctx, d_q + b * nqb, d_pos, nf, d_qsub));
        SD_CUDA(cudaStreamSynchronize(st));  // pos is a pageable host vector
        SD_TRY(fallback(ctx, dX + b * T * ld, T, n, ld, d_qsub, nf, d_osub));
        bm_scatter_kernel<<<(unsigned)ceil_div(nf, 256), 256, 0, st>>>(d_osub, d_pos, nf, d_out + b * nqb);
        ctx->last.launches++;
        SD_CUDA(cudaGetLastError());
    }
    return SD_OK;
}

// d_out[nq] = strict J=2 numerators.  Queries the matcher cannot certify are recomputed with `fallback`;
// *n_fallback counts them.
int bd_strict_match_device(sd_ctx *ctx, const double *dX, i64 T, i64 n, i64 ld, const i64 *d_q, i64 nq, i64 *d_out,
                           StrictFallback fallback, i64 *n_fallback) {
    cudaStream_t st = ctx->stream;
    if (n_fallback) *n_fallback = 0;
    if (nq == 0) return SD_OK;
    const i64 m = n - 1;
    const i64 W = ceil_div(T, 32);
    const size_t per_q = (size_t)W * m * sizeof(uint2) + (size_t)m * (sizeof(ulonglong2) + 1) + 64;
    i64 QB = (i64)((2ull << 30) / per_q);
    if (QB < BM_SQ) QB = BM_SQ;
    if (QB > 32768) QB = 32768;
    if (QB > nq) QB = nq;
    // signatures from packed ranks; very long series or few queries keep the float64 signature kernel (the rank
    // matrix would not pay)
    const bool by_ranks = T * n <= (1ll << 26) && nq >= 64;
    u32 *Rp = nullptr;
    if (by_ranks) SD_TRY(packed_ranks(ctx, dX, ld, 1, T, n, &Rp));
    // signature / flag storage borrows rank-pipeline buffers (after the rank pass, stream ordered)
    SD_TRY(ctx->buf[BUF_MASK].reserve((size_t)QB * W * m * sizeof(uint2)));
    SD_TRY(ctx->buf[BUF_PART_X].reserve((size_t)QB * m * sizeof(ulonglong2) + (size_t)QB * m + (size_t)nq + 64));
    uint2 *Mw = ctx->buf[BUF_MASK].as<uint2>();
    ulonglong2 *sig = ctx->buf[BUF_PART_X].as<ulonglong2>();
    unsigned char *tf = reinterpret_cast<unsigned char *>(sig + (size_t)QB * m);
    unsigned char *flag = tf + (size_t)QB * m;  // nq flags
    for (i64 q0 = 0; q0 < nq; q0 += QB) {
        const int nqb = (int)(nq - q0 < QB ? nq - q0 : QB);
        const dim3 sgrid((unsigned)ceil_div(n, 128), (unsigned)ceil_div(nqb, BM_SQ));
        SD_TRY(prof_begin(ctx, SD_PHASE_BD_MASKS));
        if (by_ranks)
            bd_sig_rank_kernel<<<sgrid, 128, 0, st>>>(Rp, T, n, d_q + q0, nqb, (int)W, Mw, sig, tf);
        else
            bd_sig_kernel<<<sgrid, 128, 0, st>>>(dX, T, n, ld, d_q + q0, nqb, (int)W, Mw, sig, tf, ctx->d_status);
        SD_TRY(prof_end(ctx));
        SD_TRY(prof_begin(ctx, SD_PHASE_BD_PAIRS));
        SD_TRY(launch_match(st, dim3((unsigned)nqb, 1), m, Mw, sig, tf, T, (int)W, d_out + q0, flag + q0));
        SD_TRY(prof_end(ctx));
        ctx->last.launches += 2;
        SD_CUDA(cudaGetLastError());
    }
    return recompute_flagged(ctx, dX, 1, T, n, ld, d_q, nq, flag, d_out, fallback, n_fallback);
}

// Strict J = 2 numerators of nb equally shaped matrices (dXg = [nb][T][n], nqb queries each: d_ql[nb][nqb] are
// positions inside their matrix).  One rank pass, one pack, and one signature + one match launch per chunk of
// matrices instead of ~9 launches and two host synchronisations per matrix (permutation tests).
int bd_strict_match_batched_device(sd_ctx *ctx, const double *dXg, i64 nb, i64 T, i64 n, const i64 *d_ql, i64 nqb,
                                   i64 *d_out, StrictFallback fallback) {
    cudaStream_t st = ctx->stream;
    if (nb == 0 || nqb == 0) return SD_OK;
    const i64 m = n - 1;
    const i64 W = ceil_div(T, 32), TP = W * 16;
    u32 *Rp = nullptr;
    SD_TRY(packed_ranks(ctx, dXg, n, nb, T, n, &Rp));
    const size_t per_b = (size_t)nqb * ((size_t)W * m * sizeof(uint2) + (size_t)m * (sizeof(ulonglong2) + 1));
    i64 CB = (i64)((3ull << 29) / (per_b > 0 ? per_b : 1));  // matrices per launch pair: ~1.5 GB of sign words
    if (CB < 1) CB = 1;
    if (CB > nb) CB = nb;
    if (CB > 65535) CB = 65535;
    SD_TRY(ctx->buf[BUF_MASK].reserve((size_t)CB * nqb * W * m * sizeof(uint2)));
    SD_TRY(ctx->buf[BUF_PART_X].reserve((size_t)CB * nqb * m * (sizeof(ulonglong2) + 1) + (size_t)nb * nqb + 64));
    uint2 *Mw = ctx->buf[BUF_MASK].as<uint2>();
    ulonglong2 *sig = ctx->buf[BUF_PART_X].as<ulonglong2>();
    unsigned char *tf = reinterpret_cast<unsigned char *>(sig + (size_t)CB * nqb * m);
    unsigned char *flag = tf + (size_t)CB * nqb * m;  // nb * nqb flags
    for (i64 b0 = 0; b0 < nb; b0 += CB) {
        const i64 cb = nb - b0 < CB ? nb - b0 : CB;
        SD_TRY(prof_begin(ctx, SD_PHASE_BD_MASKS));
        bd_sig_rank_kernel<<<dim3((unsigned)ceil_div(n, 128), (unsigned)ceil_div(nqb, BM_SQ), (unsigned)cb), 128, 0,
                             st>>>(Rp + b0 * TP * n, T, n, d_ql + b0 * nqb, (int)nqb, (int)W, Mw, sig, tf);
        SD_TRY(prof_end(ctx));
        SD_TRY(prof_begin(ctx, SD_PHASE_BD_PAIRS));
        SD_TRY(launch_match(st, dim3((unsigned)nqb, (unsigned)cb), m, Mw, sig, tf, T, (int)W, d_out + b0 * nqb,
                            flag + b0 * nqb));
        SD_TRY(prof_end(ctx));
        ctx->last.launches += 2;
        SD_CUDA(cudaGetLastError());
    }
    return recompute_flagged(ctx, dXg, nb, T, n, n, d_ql, nqb, flag, d_out, fallback, nullptr);
}

}  // namespace sd
