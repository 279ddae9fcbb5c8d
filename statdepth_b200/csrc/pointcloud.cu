// pointcloud.cu -- point-cloud depths: L1, simplicial (brute-force, exact predicate), Oja; and the
// multivariate functional simplex depth, which shares the simplex predicate.
//
// Reference routines replaced (statdepth/depth/calculations/):
//   _L1_depth            _pointcloud.py:125-150
//   _pointwisedepth      _pointcloud.py:44-56   ('simplex' branch: all (d+1)-subsets of the others)
//   _oja_depth           _pointcloud.py:176-204
//   _simplex_depth       _functional.py:257-286 + _simplex_containment _containment.py:105-136
// Compiled with -fmad=false: see simplex_pred.cuh.
#include "common.cuh"
#include "simplex_pred.cuh"

namespace sd {

// ---------------------------------------------------------------------------------------------
// L1 depth: L1_LANES adjacent lanes per query point, all points streamed through shared memory.  Lane k sums
// the unit vectors of the points o = k (mod L1_LANES) in index order in float64; the partial sums are added
// at the end.  (One thread per query with sqrt and divisions repeated the reference's operations bit for bit,
// _pointcloud.py:145-146, at 12.7 ms for 50 000 points; lanes + rsqrt: 3.9 ms, <= 3e-14 relative on the depth,
// the bar is 1e-12.)
// ---------------------------------------------------------------------------------------------
constexpr int L1_TILE = 512;
constexpr int L1_MAXD = 16;
#ifndef SD_L1_LANES
#define SD_L1_LANES 4
#endif
#ifndef SD_L1_ILP
#define SD_L1_ILP 1
#endif
constexpr int L1_LANES = SD_L1_LANES;  // lanes per query (1 would keep the reference's summation order bit for bit)
constexpr int L1_ILP = SD_L1_ILP;      // points in flight per lane
constexpr int L1_THREADS = 128;

template <int D>
__global__ void __launch_bounds__(L1_THREADS) l1_kernel(const double *__restrict__ P, const i64 n, const int d_rt,
                                                        const i64 *__restrict__ q, const i64 nq,
                                                        const double denom, double *__restrict__ out) {
    extern __shared__ double s_pts[];  // L1_TILE * d
    const int d = D > 0 ? D : d_rt;
    const int part = threadIdx.x % L1_LANES;
    const i64 qi = (i64)blockIdx.x * (L1_THREADS / L1_LANES) + threadIdx.x / L1_LANES;
    const bool active = qi < nq;
    const i64 p = active ? (q ? q[qi] : qi) : 0;
    double xp[D > 0 ? D : L1_MAXD], s[D > 0 ? D : L1_MAXD];
#pragma unroll
    for (int c = 0; c < (D > 0 ? D : L1_MAXD); ++c) {
        xp[c] = (c < d) ? P[p * d + c] : 0.0;
        s[c] = 0.0;
    }
    for (i64 t0 = 0; t0 < n; t0 += L1_TILE) {
        const int len = (n - t0) < L1_TILE ? (int)(n - t0) : L1_TILE;
        __syncthreads();
        for (int i = threadIdx.x; i < len * d; i += blockDim.x) s_pts[i] = P[t0 * d + i];
        __syncthreads();
        if (active) {
            // L1_ILP points at a time: their square roots and divisions are independent and overlap; the terms
            // are then added strictly in index order (adding +0.0 for the point itself changes no bit)
            for (int o0 = part * L1_ILP; o0 < len; o0 += L1_LANES * L1_ILP) {
                double term[L1_ILP][D > 0 ? D : L1_MAXD];
#pragma unroll
                for (int u = 0; u < L1_ILP; ++u) {
                    const int o = o0 + u;
                    const bool skip = o >= len || t0 + o == p;
                    double nrm2 = 0.0, diff[D > 0 ? D : L1_MAXD];
#pragma unroll
                    for (int c = 0; c < (D > 0 ? D : L1_MAXD); ++c) {
                        diff[c] = 0.0;
                        if (c < d && o < len) {
                            const double xo = s_pts[o * d + c];
                            diff[c] = xo - xp[c];
                            const double back = xp[c] - xo;
                            nrm2 += back * back;
                        }
                    }
                    // one reciprocal square root per pair instead of a square root and d divisions (<= 2 ulp per
                    // term; duplicates: 0 * inf = NaN propagates like the reference's 0 / 0)
                    const double inv = rsqrt(nrm2);
#pragma unroll
                    for (int c = 0; c < (D > 0 ? D : L1_MAXD); ++c)
                        term[u][c] = skip ? 0.0 : diff[c] * inv;
                }
#pragma unroll
                for (int u = 0; u < L1_ILP; ++u)
#pragma unroll
                    for (int c = 0; c < (D > 0 ? D : L1_MAXD); ++c)
                        if (c < d) s[c] += term[u][c];
            }
        }
    }
    double tot = 0.0;
#pragma unroll
    for (int c = 0; c < (D > 0 ? D : L1_MAXD); ++c) {
        if (c < d) {
            double v = s[c];
#pragma unroll
            for (int m = 1; m < L1_LANES; m <<= 1) v += __shfl_xor_sync(0xffffffffu, v, m);
            tot += v * v;
        }
    }
    if (active && part == 0) out[qi] = 1.0 - sqrt(tot) / denom;
}

// The others are the first n points, skipping the query when it is one of them.  n_pop = population size of the
// divisor: n for queries among the points, n + 1 for out-of-sample queries (ids >= n, never skipped).
int l1_device(sd_ctx *ctx, const double *dP, i64 n, int d, const i64 *d_q, i64 nq, double *d_out, i64 n_pop) {
    if (nq == 0) return SD_OK;
    const double denom = (double)(n_pop > 0 ? n_pop : n);
    const unsigned grid = (unsigned)ceil_div(nq, L1_THREADS / L1_LANES);
    const size_t smem = (size_t)L1_TILE * d * sizeof(double);
    cudaStream_t st = ctx->stream;
    switch (d) {
        case 1: l1_kernel<1><<<grid, L1_THREADS, smem, st>>>(dP, n, d, d_q, nq, denom, d_out); break;
        case 2: l1_kernel<2><<<grid, L1_THREADS, smem, st>>>(dP, n, d, d_q, nq, denom, d_out); break;
        case 3: l1_kernel<3><<<grid, L1_THREADS, smem, st>>>(dP, n, d, d_q, nq, denom, d_out); break;
        default:
            SD_CUDA(cudaFuncSetAttribute(l1_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         L1_TILE * L1_MAXD * (int)sizeof(double)));
            l1_kernel<0><<<grid, L1_THREADS, smem, st>>>(dP, n, d, d_q, nq, denom, d_out);
            break;
    }
    ctx->last.launches++;
    SD_CUDA(cudaGetLastError());
    return SD_OK;
}

// ---------------------------------------------------------------------------------------------
// helpers: pair unranking and block reductions
// ---------------------------------------------------------------------------------------------
// pid in [0, m(m-1)/2) -> (a < b), pid = b(b-1)/2 + a
__device__ __forceinline__ void unrank_pair(const i64 pid, i64 &a, i64 &b) {
    b = (i64)((1.0 + sqrt(1.0 + 8.0 * (double)pid)) * 0.5);
    while (b * (b - 1) / 2 > pid) --b;
    while ((b + 1) * b / 2 <= pid) ++b;
    a = pid - b * (b - 1) / 2;
}

__device__ __forceinline__ u64 block_sum_u64(u64 v, u64 *s_scratch) {
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) v += __shfl_xor_sync(0xffffffffu, v, s);
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    __syncthreads();
    if (lane == 0) s_scratch[wid] = v;
    __syncthreads();
    u64 tot = 0;
    if (threadIdx.x == 0)
        for (int w = 0; w < (int)(blockDim.x + 31) / 32; ++w) tot += s_scratch[w];
    return tot;  // valid on thread 0
}

__device__ __forceinline__ double block_sum_f64(double v, double *s_scratch) {
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) v += __shfl_xor_sync(0xffffffffu, v, s);
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    __syncthreads();
    if (lane == 0) s_scratch[wid] = v;
    __syncthreads();
    double tot = 0.0;
    if (threadIdx.x == 0)
        for (int w = 0; w < (int)(blockDim.x + 31) / 32; ++w) tot += s_scratch[w];
    return tot;
}

// ---------------------------------------------------------------------------------------------
// simplicial depth numerator: one CTA per query point, threads stride over pairs of the other
// points (positions in the "others" list skip the query), inner loops add the remaining vertices
// ---------------------------------------------------------------------------------------------
template <int D>
__global__ void __launch_bounds__(256) simplicial_kernel(const double *__restrict__ P, const i64 n,
                                                         const i64 *__restrict__ q, const double tol,
                                                         i64 *__restrict__ out) {
    __shared__ u64 s_red[8];
    const i64 p = q ? q[blockIdx.x] : (i64)blockIdx.x;
    const i64 m = n - 1;  // others
    double xp[D];
#pragma unroll
    for (int c = 0; c < D; ++c) xp[c] = P[p * D + c];
    u64 count = 0;
    const i64 npairs = m * (m - 1) / 2;
    for (i64 pid = threadIdx.x; pid < npairs; pid += blockDim.x) {
        i64 ia, ib;
        unrank_pair(pid, ia, ib);
        const i64 a = ia + (ia >= p), b = ib + (ib >= p);
        double V[(D + 1) * D];
#pragma unroll
        for (int c = 0; c < D; ++c) {
            V[c] = P[a * D + c];
            V[D + c] = P[b * D + c];
        }
        if (D == 1) {
            count += in_simplex<D>(V, xp, tol);
        } else {
            for (i64 ic = ib + 1; ic < m; ++ic) {
                const i64 c3 = ic + (ic >= p);
#pragma unroll
                for (int c = 0; c < D; ++c) V[2 * D + c] = P[c3 * D + c];
                if (D == 2) {
                    count += in_simplex<D>(V, xp, tol);
                } else {
                    for (i64 ie = ic + 1; ie < m; ++ie) {
                        const i64 c4 = ie + (ie >= p);
#pragma unroll
                        for (int c = 0; c < D; ++c) V[3 * D + c] = P[c4 * D + c];
                        count += in_simplex<D>(V, xp, tol);
                    }
                }
            }
        }
    }
    const u64 tot = block_sum_u64(count, s_red);
    if (threadIdx.x == 0) out[blockIdx.x] = (i64)tot;
}

// samples up to this size are enumerated; larger 2-D samples are counted in O(n log n) per query
// (simplicial_count.cu).  Both honour the tolerance band `tol` of the reference's LP.
constexpr i64 SIMPLICIAL_ENUM_MAX_N = 64;
constexpr i64 SIMPLEX_ENUM_MAX_N = 64;

// oos: the queries (ids >= n - 1) are not among the first n - 1 points, which are all the others (out-of-sample
// depth of a point appended to a sample of n - 1).  The enumeration kernel needs nothing else: its others are
// positions 0 .. n - 2 shifted past the query, and no position reaches a query id.  n is the population size
// either way, so both forms switch to counting at the same size.
int simplicial_device(sd_ctx *ctx, const double *dP, i64 n, int d, const i64 *d_q, i64 nq, double tol,
                      i64 *d_out, bool oos) {
    if (nq == 0) return SD_OK;
    if (d == 2 && (ctx->simplicial_impl == SD_SIMPLICIAL_COUNT ||
                   (ctx->simplicial_impl == SD_SIMPLICIAL_AUTO && n > SIMPLICIAL_ENUM_MAX_N)))
        return oos ? simplicial2_count_device(ctx, dP, n - 1, 2, 1, d_q, nq, tol, d_out, n - 1)
                   : simplicial2_count_device(ctx, dP, n, 2, 1, d_q, nq, tol, d_out);
    cudaStream_t st = ctx->stream;
    const unsigned grid = (unsigned)nq;
    switch (d) {
        case 1: simplicial_kernel<1><<<grid, 256, 0, st>>>(dP, n, d_q, tol, d_out); break;
        case 2: simplicial_kernel<2><<<grid, 256, 0, st>>>(dP, n, d_q, tol, d_out); break;
        case 3: simplicial_kernel<3><<<grid, 256, 0, st>>>(dP, n, d_q, tol, d_out); break;
        default: set_error("simplicial depth: d=%d not supported", d); return SD_ERR_UNSUPPORTED;
    }
    ctx->last.launches++;
    SD_CUDA(cudaGetLastError());
    return SD_OK;
}

// ---------------------------------------------------------------------------------------------
// Oja: sum over d-subsets of pool \ {p} of |det| / d!
// ---------------------------------------------------------------------------------------------
template <int D>
__global__ void __launch_bounds__(256) oja_kernel(const double *__restrict__ P, const i64 *__restrict__ q,
                                                  const i64 *__restrict__ pool, const i64 npool,
                                                  const double hull_volume, double *__restrict__ out) {
    __shared__ double s_red[8];
    const i64 p = q ? q[blockIdx.x] : (i64)blockIdx.x;
    double xp[D];
#pragma unroll
    for (int c = 0; c < D; ++c) xp[c] = P[p * D + c];
    double acc = 0.0;
    const i64 npairs = npool * (npool - 1) / 2;
    for (i64 pid = threadIdx.x; pid < npairs; pid += blockDim.x) {
        i64 ia, ib;
        unrank_pair(pid, ia, ib);
        const i64 a = pool ? pool[ia] : ia, b = pool ? pool[ib] : ib;
        if (a == p || b == p) continue;
        if (D == 2) {
            acc += fabs(orient2(P + a * 2, P + b * 2, xp)) / 2.0;
        } else {
            for (i64 ic = ib + 1; ic < npool; ++ic) {
                const i64 c3 = pool ? pool[ic] : ic;
                if (c3 == p) continue;
                acc += fabs(orient3(P + a * 3, P + b * 3, P + c3 * 3, xp)) / 6.0;
            }
        }
    }
    const double tot = block_sum_f64(acc, s_red);
    if (threadIdx.x == 0) out[blockIdx.x] = tot / hull_volume;
}

// pool-relative inputs of the counting path: the pool's points, and each query's position inside the pool
// (-1 if it is not a member; the reference only ever passes pool == queries, _pointcloud.py:182-193)
__global__ void oja_gather_kernel(const double *__restrict__ P, const i64 *__restrict__ pool, const i64 npool,
                                  const i64 *__restrict__ q, const i64 nq, double *__restrict__ pts,
                                  i64 *__restrict__ qpos) {
    const i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < npool) {
        const i64 s = pool ? pool[i] : i;
        pts[2 * i] = P[2 * s];
        pts[2 * i + 1] = P[2 * s + 1];
    }
    if (i < nq) {
        const i64 want = q ? q[i] : i;
        i64 pos = -1;
        if (!pool) pos = want;
        else if (i < npool && pool[i] == want) pos = i;
        else
            for (i64 k = 0; k < npool; ++k)
                if (pool[k] == want) { pos = k; break; }
        qpos[i] = pos;
    }
}

__global__ void oja_check_members_kernel(const i64 *__restrict__ qpos, const i64 nq, int *__restrict__ flag) {
    const i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < nq && qpos[i] < 0) atomicOr(flag, 1);
}

constexpr i64 OJA_ENUM_MAX_N = 256;

int oja_device(sd_ctx *ctx, const double *dP, i64 n, int d, const i64 *d_q, i64 nq, const i64 *d_pool, i64 npool,
               double hull_volume, double *d_out) {
    (void)n;
    if (nq == 0) return SD_OK;
    cudaStream_t st = ctx->stream;
    if (d == 2 && (ctx->simplicial_impl == SD_SIMPLICIAL_COUNT ||
                   (ctx->simplicial_impl == SD_SIMPLICIAL_AUTO && npool > OJA_ENUM_MAX_N))) {
        // O(n log n) per query; queries that are not pool members keep the enumeration (never the case for
        // the reference's call pattern)
        SD_TRY(ctx->buf[BUF_GEOM].reserve((size_t)npool * 2 * sizeof(double) + (size_t)nq * sizeof(i64) + 64));
        double *pts = ctx->buf[BUF_GEOM].as<double>();
        i64 *qpos = reinterpret_cast<i64 *>(pts + 2 * npool);
        int *flag = ctx->d_status + 4;  // [0..3] belong to the status word and the rank pipeline
        SD_CUDA(cudaMemsetAsync(flag, 0, sizeof(int), st));
        const i64 m = npool > nq ? npool : nq;
        oja_gather_kernel<<<(unsigned)ceil_div(m, 256), 256, 0, st>>>(dP, d_pool, npool, d_q, nq, pts, qpos);
        oja_check_members_kernel<<<(unsigned)ceil_div(nq, 256), 256, 0, st>>>(qpos, nq, flag);
        ctx->last.launches += 2;
        int h_flag = 0;
        SD_CUDA(cudaMemcpyAsync(&h_flag, flag, sizeof(int), cudaMemcpyDeviceToHost, st));
        SD_CUDA(cudaStreamSynchronize(st));
        if (!h_flag) return oja2_count_device(ctx, pts, npool, qpos, nq, hull_volume, d_out);
    }
    if (d == 2) oja_kernel<2><<<(unsigned)nq, 256, 0, st>>>(dP, d_q, d_pool, npool, hull_volume, d_out);
    else if (d == 3) oja_kernel<3><<<(unsigned)nq, 256, 0, st>>>(dP, d_q, d_pool, npool, hull_volume, d_out);
    else { set_error("oja: d=%d not supported", d); return SD_ERR_UNSUPPORTED; }
    ctx->last.launches++;
    SD_CUDA(cudaGetLastError());
    return SD_OK;
}

// ---------------------------------------------------------------------------------------------
// Blocks: B small sub-clouds of one cloud, ONE query each, in one launch.  This is what K-sampled point-cloud
// depth is made of (_samplepointwisedepth, _pointcloud.py:97-123: len(to_compute) * ss blocks of ss or ss + 1
// sampled points, each a single-query depth); the members of block b are member[off[b] .. off[b+1]) (ids into P,
// in the order the reference holds them: the L1 sum runs in that order), its query is member[off[b] + qpos[b]].
// One CTA per block; the sub-cloud is staged in shared memory when it fits.
//   kind 0: simplicial count (as a double; exact below 2^53)   kind 1: L1 depth   kind 2: Oja sum / volume[b]
// ---------------------------------------------------------------------------------------------
constexpr int BLK_SMEM_DOUBLES = 4096;  // 32 KB: sub-clouds of up to 4096 / d points are staged

template <int D>
__global__ void __launch_bounds__(256) cloud_blocks_kernel(const double *__restrict__ P, const i64 *__restrict__ member,
                                                           const i64 *__restrict__ off, const i64 *__restrict__ qpos,
                                                           const int kind, const double tol,
                                                           const double *__restrict__ volume, double *__restrict__ out) {
    __shared__ double s_pts[BLK_SMEM_DOUBLES];
    __shared__ u64 s_red[8];
    __shared__ double s_redf[8];
    const i64 b = blockIdx.x;
    const i64 m0 = off[b], m = off[b + 1] - m0;  // members of this block
    const i64 pq = qpos[b];
    if (m * D > BLK_SMEM_DOUBLES) {  // host side refuses these; keep the kernel total
        if (threadIdx.x == 0) out[b] = nan("");
        return;
    }
    for (i64 i = threadIdx.x; i < m * D; i += blockDim.x) s_pts[i] = P[member[m0 + i / D] * D + i % D];
    __syncthreads();
    double xp[D];
#pragma unroll
    for (int c = 0; c < D; ++c) xp[c] = s_pts[pq * D + c];
    if (kind == 1) {
        // sequential sum in member order by ONE thread per coordinate would be the reference bit for bit; the blocks
        // are small, so thread 0 does exactly that (sqrt and divisions as in _L1_depth, _pointcloud.py:145-146)
        if (threadIdx.x == 0) {
            double sum[D];
#pragma unroll
            for (int c = 0; c < D; ++c) sum[c] = 0.0;
            for (i64 o = 0; o < m; ++o) {
                if (o == pq) continue;
                double nrm2 = 0.0, diff[D];
#pragma unroll
                for (int c = 0; c < D; ++c) {
                    diff[c] = s_pts[o * D + c] - xp[c];
                    const double back = xp[c] - s_pts[o * D + c];
                    nrm2 += back * back;
                }
                const double nrm = sqrt(nrm2);
#pragma unroll
                for (int c = 0; c < D; ++c) sum[c] += diff[c] / nrm;
            }
            double tot = 0.0;
#pragma unroll
            for (int c = 0; c < D; ++c) tot += sum[c] * sum[c];
            out[b] = 1.0 - sqrt(tot) / (double)m;
        }
        return;
    }
    const i64 mo = m - 1;  // others; position i of the "others" list skips the query
    const i64 npairs = mo * (mo - 1) / 2;
    u64 count = 0;
    double acc = 0.0;
    for (i64 pid = threadIdx.x; pid < npairs; pid += blockDim.x) {
        i64 ia, ib;
        unrank_pair(pid, ia, ib);
        const i64 a = ia + (ia >= pq), bb = ib + (ib >= pq);
        if (kind == 2) {
            if (D == 2) {
                acc += fabs(orient2(s_pts + a * 2, s_pts + bb * 2, xp)) / 2.0;
            } else if (D == 3) {
                for (i64 ic = ib + 1; ic < mo; ++ic) {
                    const i64 c3 = ic + (ic >= pq);
                    acc += fabs(orient3(s_pts + a * 3, s_pts + bb * 3, s_pts + c3 * 3, xp)) / 6.0;
                }
            }
            continue;
        }
        double V[(D + 1) * D];
#pragma unroll
        for (int c = 0; c < D; ++c) {
            V[c] = s_pts[a * D + c];
            V[D + c] = s_pts[bb * D + c];
        }
        if (D == 1) {
            count += in_simplex<D>(V, xp, tol);
        } else {
            for (i64 ic = ib + 1; ic < mo; ++ic) {
                const i64 c3 = ic + (ic >= pq);
#pragma unroll
                for (int c = 0; c < D; ++c) V[2 * D + c] = s_pts[c3 * D + c];
                if (D == 2) {
                    count += in_simplex<D>(V, xp, tol);
                } else {
                    for (i64 ie = ic + 1; ie < mo; ++ie) {
                        const i64 c4 = ie + (ie >= pq);
#pragma unroll
                        for (int c = 0; c < D; ++c) V[3 * D + c] = s_pts[c4 * D + c];
                        count += in_simplex<D>(V, xp, tol);
                    }
                }
            }
        }
    }
    if (kind == 2) {
        const double tot = block_sum_f64(acc, s_redf);
        if (threadIdx.x == 0) out[b] = tot / volume[b];
    } else {
        const u64 tot = block_sum_u64(count, s_red);
        if (threadIdx.x == 0) out[b] = (double)tot;
    }
}

int cloud_blocks_device(sd_ctx *ctx, const double *dP, int d, const i64 *d_member, const i64 *d_off,
                        const i64 *d_qpos, i64 B, int kind, double tol, const double *d_volume, double *d_out) {
    if (B == 0) return SD_OK;
    cudaStream_t st = ctx->stream;
    const unsigned grid = (unsigned)B;
    switch (d) {
        case 1: cloud_blocks_kernel<1><<<grid, 256, 0, st>>>(dP, d_member, d_off, d_qpos, kind, tol, d_volume, d_out); break;
        case 2: cloud_blocks_kernel<2><<<grid, 256, 0, st>>>(dP, d_member, d_off, d_qpos, kind, tol, d_volume, d_out); break;
        case 3: cloud_blocks_kernel<3><<<grid, 256, 0, st>>>(dP, d_member, d_off, d_qpos, kind, tol, d_volume, d_out); break;
        default: set_error("point-cloud blocks: d=%d not supported (1..3)", d); return SD_ERR_UNSUPPORTED;
    }
    ctx->last.launches++;
    SD_CUDA(cudaGetLastError());
    return SD_OK;
}

// ---------------------------------------------------------------------------------------------
// multivariate functional simplex depth numerator: one CTA per query curve; F[(i*T + t)*D + c]
// ---------------------------------------------------------------------------------------------
template <int D>
__device__ __forceinline__ i64 subset_count(const double *__restrict__ F, const i64 T, const i64 qc, const i64 *o,
                                            const bool relax, const double tol) {
    i64 cnt = 0;
    for (i64 t = 0; t < T; ++t) {
        double V[(D + 1) * D], xp[D];
#pragma unroll
        for (int k = 0; k <= D; ++k)
#pragma unroll
            for (int c = 0; c < D; ++c) V[k * D + c] = F[(o[k] * T + t) * D + c];
#pragma unroll
        for (int c = 0; c < D; ++c) xp[c] = F[(qc * T + t) * D + c];
        if (in_simplex<D>(V, xp, tol)) ++cnt;
        else if (!relax) return 0;
    }
    return relax ? cnt : 1;  // strict: reached the end <=> contained at all T rows
}

template <int D>
__global__ void __launch_bounds__(256) simplex_depth_kernel(const double *__restrict__ F, const i64 N, const i64 T,
                                                            const i64 *__restrict__ q, const int relax,
                                                            const double tol, i64 *__restrict__ out) {
    __shared__ u64 s_red[8];
    const i64 qc = q ? q[blockIdx.x] : (i64)blockIdx.x;
    const i64 m = N - 1;
    u64 acc = 0;
    const i64 npairs = m * (m - 1) / 2;
    for (i64 pid = threadIdx.x; pid < npairs; pid += blockDim.x) {
        i64 ia, ib;
        unrank_pair(pid, ia, ib);
        i64 o[4];
        o[0] = ia + (ia >= qc);
        o[1] = ib + (ib >= qc);
        o[2] = o[3] = 0;
        if (D == 1) {
            acc += (u64)subset_count<D>(F, T, qc, o, relax != 0, tol);
        } else {
            for (i64 ic = ib + 1; ic < m; ++ic) {
                o[2] = ic + (ic >= qc);
                if (D == 2) {
                    acc += (u64)subset_count<D>(F, T, qc, o, relax != 0, tol);
                } else {
                    for (i64 ie = ic + 1; ie < m; ++ie) {
                        o[3] = ie + (ie >= qc);
                        acc += (u64)subset_count<D>(F, T, qc, o, relax != 0, tol);
                    }
                }
            }
        }
    }
    const u64 tot = block_sum_u64(acc, s_red);
    if (threadIdx.x == 0) out[blockIdx.x] = (i64)tot;
}

// ---------------------------------------------------------------------------------------------
// Strict multivariate simplex depth, d = 2, for samples the plain enumeration above cannot finish (BASELINE
// config 4: 5 000 curves x 256 points -> C(4999,3) = 2.1e10 triples per query).  A triple counts iff the query lies
// in its closed triangle (tolerance band tol) at ALL T rows, so every row prunes: the directions v_o = x_o - x_q of
// the first SX_ROWS rows are staged in shared memory as floats (x, y and an upper bound r of |v_o|: 12 bytes per
// curve and row, 180 KB at N = 5000), every thread takes pairs (a, b) and streams c > b through two float cross
// products per staged row.  With e_k = the three edge functions of the triangle seen from the query,
//     all e_k  >  +eps_k                          -> inside at this row for certain (any tolerance)
//     some e_k < -tol (r_i + r_j) - eps_k         -> farther than tol from that edge's line: outside for certain
// (|x_i - x_j| <= |v_i| + |v_j|; eps_k = 1e-6 r_i r_j covers the float rounding of v and of the cross product, 1e-12
// r_i r_j for the float64 rows), and only the rest -- within the band of an edge, or degenerate -- is decided by the
// reference predicate in_simplex<2> itself on the float64 vertices.  A triple survives a row with probability
// <= 1/4 on average, so 1.6 % reach the remaining rows, which are walked in float64 through L2 with early exit (the
// first version staged one row only and spent its time on the 25 % survivors' L2 reads: 312 ms per query).
// Decisions are exactly those of the enumeration kernel / the oracle.
// ---------------------------------------------------------------------------------------------
#ifndef SD_SX_THREADS
#define SD_SX_THREADS 512
#endif
constexpr int SX_THREADS = SD_SX_THREADS;
constexpr int SX_ROWS = 3;

// +1 inside for certain, -1 outside for certain, 0 ask the predicate.  kE: relative rounding bound of the e's.
template <typename R>
__device__ __forceinline__ int sx_classify(const R e0, const R e1, const R e2, const R ra, const R rb, const R rc,
                                           const R tol, const R kE) {
    const R pab = ra * rb, pbc = rb * rc, pca = rc * ra;
    const bool pos = e0 > kE * pab && e1 > kE * pbc && e2 > kE * pca;
    const bool neg = e0 < -kE * pab && e1 < -kE * pbc && e2 < -kE * pca;
    if (pos || neg) return 1;
    // orientation of the triangle = sign of e0 + e1 + e2; an edge function of the opposite sign, beyond the band
    const R D = (e0 + e1) + e2, big = (R)3 * kE * (pab + pbc + pca), up = (R)1 + (R)1e-6;
    const R m0 = tol * (ra + rb) * up + kE * pab, m1 = tol * (rb + rc) * up + kE * pbc, m2 = tol * (rc + ra) * up + kE * pca;
    if (D > big && (e0 < -m0 || e1 < -m1 || e2 < -m2)) return -1;
    if (D < -big && (e0 > m0 || e1 > m1 || e2 > m2)) return -1;
    return 0;
}

// row t of triple (oa, ob, oc) in float64: certain cases by the edge functions, the rest by the predicate
__device__ __forceinline__ bool sx_row64(const double *__restrict__ F, const i64 T, const i64 t, const i64 oa,
                                         const i64 ob, const i64 oc, const double px, const double py,
                                         const double tol) {
    const double ax = F[(oa * T + t) * 2], ay = F[(oa * T + t) * 2 + 1];
    const double bx = F[(ob * T + t) * 2], by = F[(ob * T + t) * 2 + 1];
    const double cx = F[(oc * T + t) * 2], cy = F[(oc * T + t) * 2 + 1];
    const double vax = ax - px, vay = ay - py, vbx = bx - px, vby = by - py, vcx = cx - px, vcy = cy - py;
    const double f0 = vax * vby - vay * vbx, f1 = vbx * vcy - vby * vcx, f2 = vcx * vay - vcy * vax;
    // |v| <= |vx| + |vy|: an upper bound without square roots
    const int c2 = sx_classify<double>(f0, f1, f2, fabs(vax) + fabs(vay), fabs(vbx) + fabs(vby), fabs(vcx) + fabs(vcy),
                                       tol, 1e-12);
    if (c2) return c2 > 0;
    const double V[6] = {ax, ay, bx, by, cx, cy}, P2[2] = {px, py};
    return in_simplex<2>(V, P2, tol);
}

// Survivors are not followed inline -- one surviving lane would hold its 31 neighbours through rows they have
// already failed (with a quarter surviving per row, SOME lane of a warp nearly always survives) -- but COMPACTED:
// a warp appends the triples that passed row 0 to a small queue in shared memory (ballot + prefix), and whenever
// 32 are waiting it runs them through the other staged rows, one triple per lane; what passes those is queued
// again and walks the float64 rows 32 at a time.  (inline: 180 ms per query at config-4 size.)
struct SxQueue {
    ushort4 *slot;  // [64] (ia, ib, ic, unsure-row bits)
    int count;      // warp-uniform
};

__device__ __forceinline__ void sx_push(SxQueue &Q, const bool put, const ushort4 e, const int lane) {
    const u32 mask = __ballot_sync(0xffffffffu, put);
    if (put) Q.slot[Q.count + __popc(mask & ((1u << lane) - 1u))] = e;
    Q.count += __popc(mask);
    __syncwarp();
}

__global__ void __launch_bounds__(SX_THREADS) simplex2_strict_kernel(const double *__restrict__ F, const i64 N, const i64 T,
                                                                     const i64 *__restrict__ q, const double tol,
                                                                     i64 *__restrict__ out) {
    extern __shared__ __align__(16) unsigned char sx_smem[];
    const i64 m = N - 1;
    const int nr = T < SX_ROWS ? (int)T : SX_ROWS;           // staged rows
    double *pq = reinterpret_cast<double *>(sx_smem);          // [T][2] the query curve
    float2 *xy = reinterpret_cast<float2 *>(pq + 2 * T);       // [nr][m]
    float *rr = reinterpret_cast<float *>(xy + (size_t)nr * m);  // [nr][m]
    __shared__ u64 s_red[SX_THREADS / 32];
    __shared__ ushort4 s_q[SX_THREADS / 32][2][64];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const i64 qi = blockIdx.y;
    const i64 qc = q ? q[qi] : qi;
    for (i64 i = threadIdx.x; i < 2 * T; i += blockDim.x) pq[i] = F[qc * T * 2 + i];
    __syncthreads();
    for (i64 i = threadIdx.x; i < m * nr; i += blockDim.x) {
        const i64 r = i / m, k = i - r * m;
        const i64 o = k + (k >= qc);
        const double vx = F[(o * T + r) * 2] - pq[2 * r], vy = F[(o * T + r) * 2 + 1] - pq[2 * r + 1];
        xy[i] = make_float2(__double2float_rn(vx), __double2float_rn(vy));
        rr[i] = __double2float_ru((fabs(vx) + fabs(vy)) * (1.0 + 1e-6));  // upper bound of |v|, rounding included
    }
    __syncthreads();
    const float tolf = __double2float_ru(tol);
    u64 count = 0;
    SxQueue Q1 = {s_q[wid][0], 0}, Q2 = {s_q[wid][1], 0};

    // float64 rows of one queued triple per lane
    auto run64 = [&](const bool have, const ushort4 e) {
        if (!have) return;
        const i64 oa = e.x + (e.x >= qc), ob = e.y + (e.y >= qc), oc = e.z + (e.z >= qc);
        bool all = true;
        for (int r = 0; r < nr && all; ++r)  // staged rows the float test could not decide
            if (e.w & (1u << r)) all = sx_row64(F, T, r, oa, ob, oc, pq[2 * r], pq[2 * r + 1], tol);
        for (i64 t = nr; t < T && all; ++t) all = sx_row64(F, T, t, oa, ob, oc, pq[2 * t], pq[2 * t + 1], tol);
        count += all;
    };
    // staged rows 1 .. nr-1 of one queued triple per lane; survivors go to Q2
    auto run_rows = [&](const bool have, ushort4 e) {
        bool alive = have;
#pragma unroll
        for (int r = 1; r < SX_ROWS; ++r) {
            if (r < nr && alive) {
                const float2 A = xy[(size_t)r * m + e.x], B = xy[(size_t)r * m + e.y], C = xy[(size_t)r * m + e.z];
                const float e0 = A.x * B.y - A.y * B.x, e1 = B.x * C.y - B.y * C.x, e2 = C.x * A.y - C.y * A.x;
                const int cls = sx_classify<float>(e0, e1, e2, rr[(size_t)r * m + e.x], rr[(size_t)r * m + e.y],
                                                   rr[(size_t)r * m + e.z], tolf, 1e-6f);
                if (cls < 0) alive = false;
                else if (cls == 0) e.w |= (unsigned short)(1u << r);
            }
        }
        sx_push(Q2, alive, e, lane);
        if (Q2.count >= 32) {
            Q2.count -= 32;
            run64(true, Q2.slot[Q2.count + lane]);
            __syncwarp();
        }
    };

    const i64 npairs = m * (m - 1) / 2;
    const i64 stride = (i64)gridDim.x * blockDim.x;
    for (i64 base = (i64)blockIdx.x * blockDim.x + wid * 32; base < npairs; base += stride) {  // warp-uniform
        const i64 pid = base + lane;
        const bool valid = pid < npairs;
        i64 ia = 0, ib = 1;
        if (valid) unrank_pair(pid, ia, ib);
        const float2 A = xy[ia], B = xy[ib];
        const float rA = rr[ia], rB = rr[ib];
        const float e0 = A.x * B.y - A.y * B.x;
        int nc = valid ? (int)(m - ib - 1) : 0, nmax = nc;
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) nmax = max(nmax, __shfl_xor_sync(0xffffffffu, nmax, d));
        for (int k = 0; k < nmax; ++k) {
            const i64 ic = ib + 1 + k;
            bool pass = false;
            ushort4 e = make_ushort4((unsigned short)ia, (unsigned short)ib, (unsigned short)ic, 0);
            if (k < nc) {
                const float2 C = xy[ic];
                const float e1 = B.x * C.y - B.y * C.x, e2 = C.x * A.y - C.y * A.x;
                const int cls = sx_classify<float>(e0, e1, e2, rA, rB, rr[ic], tolf, 1e-6f);
                pass = cls >= 0;
                e.w = cls == 0 ? 1 : 0;
            }
            sx_push(Q1, pass, e, lane);
            if (Q1.count >= 32) {
                Q1.count -= 32;
                run_rows(true, Q1.slot[Q1.count + lane]);
                __syncwarp();
            }
        }
    }
    // drain
    run_rows(lane < Q1.count, Q1.slot[lane < Q1.count ? lane : 0]);
    Q1.count = 0;
    __syncwarp();
    while (Q2.count > 0) {
        const int take = Q2.count < 32 ? Q2.count : 32;
        Q2.count -= take;
        run64(lane < take, Q2.slot[Q2.count + (lane < take ? lane : 0)]);
        __syncwarp();
    }
    const u64 tot = block_sum_u64(count, s_red);
    if (threadIdx.x == 0 && tot) atomicAdd((u64 *)&out[qi], tot);
}

int simplex_depth_device(sd_ctx *ctx, const double *dF, i64 N, i64 T, int d, const i64 *d_q, i64 nq, int relax,
                         double tol, i64 *d_out) {
    if (nq == 0) return SD_OK;
    // relaxed depth is a sum over time points of triangle counts: countable per (query, time point)
    if (d == 2 && relax && (ctx->simplicial_impl == SD_SIMPLICIAL_COUNT ||
                            (ctx->simplicial_impl == SD_SIMPLICIAL_AUTO && N > SIMPLEX_ENUM_MAX_N)))
        return simplicial2_count_device(ctx, dF, N, 2 * T, T, d_q, nq, tol, d_out);
    cudaStream_t st = ctx->stream;
    const size_t sx_bytes = (size_t)(N - 1) * 12 * (T < SX_ROWS ? T : SX_ROWS) + (size_t)T * 2 * sizeof(double);
    if (d == 2 && !relax && N >= 4 && sx_bytes <= (size_t)(224 - SX_THREADS / 32) * 1024) {  // static: 1 KB of queues per warp
        // first-row pruning in shared memory; several CTAs per query so that a handful of queries fills the GPU
        SD_CUDA(cudaFuncSetAttribute(simplex2_strict_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sx_bytes));
        SD_CUDA(cudaMemsetAsync(d_out, 0, (size_t)nq * sizeof(i64), st));
        const i64 npairs = (N - 1) * (N - 2) / 2;
        i64 slices = ceil_div(npairs, (i64)SX_THREADS * 8);
        const i64 want = 2 * (i64)ctx->sm_count / nq;  // one resident CTA per SM: whole waves, no ragged third one
        if (slices > want) slices = want;
        if (slices < 1) slices = 1;
        for (i64 q0 = 0; q0 < nq; q0 += 65535) {
            const i64 nb = nq - q0 < 65535 ? nq - q0 : 65535;
            simplex2_strict_kernel<<<dim3((unsigned)slices, (unsigned)nb), SX_THREADS, sx_bytes, st>>>(
                dF, N, T, d_q ? d_q + q0 : nullptr, tol, d_out + q0);
            ctx->last.launches++;
        }
        SD_CUDA(cudaGetLastError());
        return SD_OK;
    }
    const unsigned grid = (unsigned)nq;
    switch (d) {
        case 1: simplex_depth_kernel<1><<<grid, 256, 0, st>>>(dF, N, T, d_q, relax, tol, d_out); break;
        case 2: simplex_depth_kernel<2><<<grid, 256, 0, st>>>(dF, N, T, d_q, relax, tol, d_out); break;
        case 3: simplex_depth_kernel<3><<<grid, 256, 0, st>>>(dF, N, T, d_q, relax, tol, d_out); break;
        default: set_error("simplex depth: d=%d not supported", d); return SD_ERR_UNSUPPORTED;
    }
    ctx->last.launches++;
    SD_CUDA(cudaGetLastError());
    return SD_OK;
}

}  // namespace sd
