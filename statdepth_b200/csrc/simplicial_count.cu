// simplicial_count.cu -- exact O(n log n) counting of the triangles that contain a query point (d = 2).
//
// Replaces the enumeration of all 3-subsets in the 'simplex' branch of _pointwisedepth
// (statdepth/depth/calculations/_pointcloud.py:44-56) and, per time point, in _simplex_depth with
// relax=True (_functional.py:257-286) when the sample is too large to enumerate (BASELINE configs 5 and
// 4: 50 000 points / 5 000 curves x 256 points).  Rousseeuw-Ruts style: a closed triangle of three other
// points does NOT contain p iff its three directions from p lie in an open half-plane, and such a triple
// has a unique first direction in counter-clockwise order.  With directions grouped into classes of
// equal angle (g points each) and c = number of points strictly inside the half-turn after the class,
//     #non-containing triples whose first class is this one = C(g + c, 3) - C(c, 3)
//     #containing = C(m, 3) - sum over classes                  (m = all other points; points equal to p
//                                                               only form containing triples)
// Angles are never computed: each direction d = x - p gets the key  8 + octant + f  in [8, 16), f the
// correctly rounded ratio of its smaller to its larger component (mirrored in odd octants).  Correct
// rounding is monotone, so the key order IS the angular order of the computed directions, directions
// that are exactly collinear get identical keys, and the antipode is exactly key +- 4 (one binade).
// Ranks come from the modified-band-depth rank pipeline (mbd.cu), run on two key matrices per batch of
// instances: A = keys (n per row), B = keys and antipodes (2n per row).
//
// Semantics.  tol == 0: exact closed triangles of the computed float64 directions (keys above).
// tol > 0 (the default, 1e-7): the reference decides with an LP (scipy.optimize.linprog, _containment.py:164-176)
// whose feasibility band accepts p up to ~1e-7 OUTSIDE a triangle, and its own multivariate fixture consists of
// collinear triples only (testing/_generating.py:94-96), so that band decides every one of them.  The
// enumeration kernels restate the LP as dist(p, triangle) <= tol (simplex_pred.cuh); the counting form of the
// same predicate: a triangle MISSES the closed disk D(p, tol) iff a tangent line of the disk has all three
// vertices strictly beyond it, i.e. iff the three open arcs
//     A_i = (phi_i - alpha_i, phi_i + alpha_i),  phi_i = angle of x_i - p,  alpha_i = acos(tol / |x_i - p|) < pi/2
// of tangent directions have a common point (points within tol of p have no arc: every triangle through them
// meets the disk).  Arcs are shorter than pi, so a non-empty common intersection is one arc whose start is
// the start s_i of exactly one class of arcs with equal start, and
//     #missing = sum over classes [C(g + c, 3) - C(c, 3)],   c = #{other arcs that contain s_i}
//              c = #{s_j < s_i} - #{e_j <= s_i} + #{arcs that wrap past 2 pi}      (e_j taken mod 2 pi)
// -- again two rank passes (starts; starts and ends) through the K1 pipeline.  With tol = 0 the arcs are
// the open half-turns of the exact formula.  Angles here come from atan2 / acos (a few ulp): decisions can
// differ from the enumeration predicate only for triangles whose distance to p is within ~1e-15 |x - p| of
// tol, far inside the documented tie band of the LP itself (DESIGN.md "Oracle and parity").
// Halfspace (Tukey) depth (K11) reduces the same keys and rank passes (tol = 0) to a minimum of half-turn counts
// instead: hs_reduce_kernel, selected by simplicial2_count_device's `reduce`.
#include "angular_key.cuh"
#include "common.cuh"

namespace sd {

constexpr double SC_TWO_PI = 6.283185307179586476925286766559;

// KA[i][j] = key_j; KB[i][j] = key_j, KB[i][n + j] = antipode of key_j.
// tol > 0: key_j = start of arc j in [0, 2 pi], second half of KB = its end mod 2 pi (sentinels as for tol = 0).
__global__ void __launch_bounds__(256) sc_keys_kernel(const ScGeom g, const i64 n, const i64 ninst, const double tol,
                                                      double *__restrict__ KA, double *__restrict__ KB,
                                                      int *__restrict__ status) {
    const i64 li = blockIdx.y;  // instance within the batch
    if (li >= ninst) return;
    const i64 inst = g.inst0 + li;
    const i64 q = sc_query(g, inst);
    const i64 off = sc_off(g, inst);
    const double px = g.pts[q * g.stride_j + off], py = g.pts[q * g.stride_j + off + 1];
    bool bad = false;
    for (i64 j = (i64)blockIdx.x * blockDim.x + threadIdx.x; j < n; j += (i64)gridDim.x * blockDim.x) {
        double u, w;
        if (j == q) {
            u = w = SC_SELF;
        } else {
            const double xj = g.pts[j * g.stride_j + off], yj = g.pts[j * g.stride_j + off + 1];
            bad |= !isfinite(xj) || !isfinite(yj);
            const double dx = xj - px, dy = yj - py;
            if (dx == 0.0 && dy == 0.0) {
                u = w = SC_ZERO;
            } else if (tol > 0.0) {
                const double r = hypot(dx, dy);
                if (r <= tol) {
                    u = w = SC_ZERO;  // within the band of p: every triangle through this point meets the disk
                } else {
                    double phi = atan2(dy, dx);
                    if (phi < 0.0) phi += SC_TWO_PI;
                    const double alpha = acos(tol / r);
                    u = phi - alpha;
                    if (u < 0.0) u += SC_TWO_PI;
                    w = u + 2.0 * alpha;
                    if (w >= SC_TWO_PI) w -= SC_TWO_PI;  // the arc wraps: its end lies below its start
                }
            } else {
                u = sc_key(dx, dy);
                w = u < 12.0 ? u + 4.0 : u - 4.0;  // exact: same binade
            }
        }
        KA[li * n + j] = u;
        KB[li * 2 * n + j] = u;
        KB[li * 2 * n + n + j] = w;
    }
    if (bad || !isfinite(px) || !isfinite(py)) atomicOr(status, ST_NONFINITE);
}

// C(m, 3), exact whenever it fits in int64: the even factor is halved and the multiple of 3 divided by 3 before the
// product, so no partial product exceeds the result ((m (m - 1) / 2) (m - 2) would wrap from m = 2 642 247).
__device__ __forceinline__ i64 c3(i64 m) {
    if (m < 3) return 0;
    i64 a = m, b = m - 1, c = m - 2;
    if (a % 2 == 0) a /= 2;
    else b /= 2;
    if (a % 3 == 0) a /= 3;
    else if (b % 3 == 0) b /= 3;
    else c /= 3;
    return a * b * c;
}

// pass 1 of the reductions, block-wide: the number of real directions m' and how many of them lie in [0, pi)
// (key < 12); ARCS: `low` counts the arcs that wrap past 2 pi (end below start).  kb_hi = second half of row B.
template <bool ARCS>
__device__ __forceinline__ void sc_count_real(const double *__restrict__ ka, const double *__restrict__ kb_hi,
                                              const i64 n, i64 *s_cnt, i64 &mreal, i64 &low_out) {
    i64 real = 0, low = 0;
    for (i64 j = threadIdx.x; j < n; j += blockDim.x) {
        const double u = ka[j];
        real += u < 16.0;
        if (ARCS) low += u < 16.0 && kb_hi[j] < u;
        else low += u < 12.0;
    }
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) {
        real += __shfl_xor_sync(0xffffffffu, real, s);
        low += __shfl_xor_sync(0xffffffffu, low, s);
    }
    if (threadIdx.x == 0) { s_cnt[0] = 0; s_cnt[1] = 0; }
    __syncthreads();
    if ((threadIdx.x & 31) == 0) {
        atomicAdd((u64 *)&s_cnt[0], (u64)real);
        atomicAdd((u64 *)&s_cnt[1], (u64)low);
    }
    __syncthreads();
    mreal = s_cnt[0];
    low_out = s_cnt[1];
}

// one CTA per instance.  bA/aA: ranks of row A; bB/aB: ranks (strictly below / above) of row B.
// out[query slot] += #triangles of other points containing the query point (ARCS: meeting the disk D(p, tol)).
template <bool ARCS>
__global__ void __launch_bounds__(256) sc_reduce_kernel(const ScGeom g, const i64 n, const double *__restrict__ KA,
                                                        const double *__restrict__ KB,
                                                        const int *__restrict__ bA, const int *__restrict__ aA,
                                                        const int *__restrict__ bB, const int *__restrict__ aB,
                                                        int *__restrict__ claim, const i64 m_others,
                                                        i64 *__restrict__ out) {
    __shared__ i64 s_red[8];
    __shared__ i64 s_cnt[2];
    const i64 li = blockIdx.x;
    const i64 inst = g.inst0 + li;
    const double *ka = KA + li * n;
    const int *ba = bA + li * n, *aa = aA + li * n, *bb = bB + li * 2 * n, *ab = aB + li * 2 * n;
    int *cl = claim + li * n;
    i64 mreal, L4;
    sc_count_real<ARCS>(ka, KB + li * 2 * n + n, n, s_cnt, mreal, L4);
    const i64 H = mreal - L4;
    // pass 2: every class of equal directions contributes C(g + c, 3) - C(c, 3) once
    i64 noncontain = 0;
    for (i64 j = threadIdx.x; j < n; j += blockDim.x) {
        const double u = ka[j];
        if (!(u < 16.0)) continue;  // zero vector or the query itself
        const i64 L = ba[j];                      // real directions strictly before this one
        const i64 gsz = n - L - (i64)aa[j];       // size of its class (sentinels are never equal to it)
        i64 c;
        if (ARCS) {
            // #{starts < s} - #{ends <= s} + #wrapping, #{ends <= s} = #{B <= s} - #{A <= s}
            c = L - ((2 * n - (i64)ab[j]) - (n - (i64)aa[j])) + L4;
        } else if (u < 12.0) {
            const i64 b2w = bb[n + j];            // entries of row B strictly below the antipode
            const i64 Lw = b2w - L - H;           // real directions strictly before the antipode
            c = Lw - L - gsz;
        } else {
            const i64 b2w = bb[n + j];
            const i64 Lw = b2w - L + L4;
            c = (mreal - L - gsz) + Lw;
        }
        if (gsz == 1) {
            noncontain += c * (c - 1) / 2;        // C(1 + c, 3) - C(c, 3) = C(c, 2)
        } else if (atomicCAS(&cl[L], 0, 1) == 0) {  // first member of the class to arrive speaks for it
            noncontain += c3(gsz + c) - c3(c);
        }
    }
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) noncontain += __shfl_xor_sync(0xffffffffu, noncontain, s);
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = noncontain;
    __syncthreads();
    if (threadIdx.x == 0) {
        i64 tot = 0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) tot += s_red[w];
        atomicAdd((u64 *)&out[inst / g.T], (u64)(c3(m_others) - tot));
    }
}

// Halfspace (Tukey) depth numerator, one CTA per instance (tolerance 0 keys only):
//     h = z + min over real directions j of min(k_j, m' - k_j),   k_j = #{real directions in (phi_j, phi_j + pi]}
// z = n - m' counts the query itself and the points equal to it; h = n when no direction is real (the min starts at
// m').  k_j = c + g_anti: c = directions strictly inside the half-turn (as the tol = 0 branch of sc_reduce_kernel),
// g_anti = entries of row B equal to the antipode (2n - bB - aB at n + j) less the g antipodes of j's own class.
// Every member of a class gives the same k and min is idempotent: no claim array.  out[inst] = h for point clouds
// (T = 1), out[inst / T] += h for curves.  A k outside [0, m'] sets ST_INTERNAL.
__global__ void __launch_bounds__(256) hs_reduce_kernel(const ScGeom g, const i64 n, const double *__restrict__ KA,
                                                        const double *__restrict__ KB,
                                                        const int *__restrict__ bA, const int *__restrict__ aA,
                                                        const int *__restrict__ bB, const int *__restrict__ aB,
                                                        i64 *__restrict__ out, int *__restrict__ status) {
    __shared__ i64 s_red[8];
    __shared__ i64 s_cnt[2];
    const i64 li = blockIdx.x;
    const i64 inst = g.inst0 + li;
    const double *ka = KA + li * n;
    const int *ba = bA + li * n, *aa = aA + li * n, *bb = bB + li * 2 * n, *ab = aB + li * 2 * n;
    i64 mreal, L4;
    sc_count_real<false>(ka, KB + li * 2 * n + n, n, s_cnt, mreal, L4);
    const i64 H = mreal - L4;
    i64 best = mreal;
    bool bad = false;
    for (i64 j = threadIdx.x; j < n; j += blockDim.x) {
        const double u = ka[j];
        if (!(u < 16.0)) continue;
        const i64 L = ba[j];
        const i64 gsz = n - L - (i64)aa[j];
        const i64 b2w = bb[n + j];
        const i64 c = u < 12.0 ? (b2w - L - H) - L - gsz : (mreal - L - gsz) + (b2w - L + L4);
        const i64 k = c + (2 * n - b2w - (i64)ab[n + j]) - gsz;
        bad |= k < 0 || k > mreal;
        const i64 side = k < mreal - k ? k : mreal - k;
        best = side < best ? side : best;
    }
    if (bad) atomicOr(status, ST_INTERNAL);
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) {
        const i64 o = __shfl_xor_sync(0xffffffffu, best, s);
        best = o < best ? o : best;
    }
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = best;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < (int)(blockDim.x >> 5); ++w) best = s_red[w] < best ? s_red[w] : best;
        const i64 h = n - mreal + best;
        if (g.T == 1) out[inst] = h;
        else atomicAdd((u64 *)&out[inst / g.T], (u64)h);
    }
}

// Counts for `nq` queries x `T` instances each (T = 1 for point clouds).  d_out[nq] is zeroed here.
// m_others < 0: the queries are among the n points (n - 1 others); m_others = n: out-of-sample queries (ids >= n,
// coordinates read from the same array), every one of the n points is an other.
// reduce: SC_TRIANGLES (sc_reduce_kernel) or SC_HALFSPACE (hs_reduce_kernel: tol = 0, in-sample queries).
int simplicial2_count_device(sd_ctx *ctx, const double *d_pts, i64 n, i64 stride_j, i64 T, const i64 *d_q, i64 nq,
                             double tol, i64 *d_out, i64 m_others, ScReduce reduce) {
    cudaStream_t st = ctx->stream;
    SD_CUDA(cudaMemsetAsync(d_out, 0, (size_t)nq * sizeof(i64), st));
    const i64 ninst_total = nq * T;
    const bool hs = reduce == SC_HALFSPACE;
    if (m_others < 0) m_others = n - 1;
    if (ninst_total == 0) return SD_OK;
    if (!hs && m_others < 3) return SD_OK;  // fewer than 3 other points: no triangle
    if (2 * n >= (1ll << 31)) {
        set_error("simplicial counting: n=%lld too large", (long long)n);
        return SD_ERR_UNSUPPORTED;
    }
    if (!(tol >= 0.0)) {
        set_error("simplicial counting: tolerance %g is negative or NaN", tol);
        return SD_ERR_INVALID;
    }
    // a triangle count is at most C(m_others, 3) per instance, and curves add T of them into one int64 (the halfspace
    // numerators are at most T n).  Exact: m_others < 2^30 here, so C(m_others, 3) < 2^90.
    if (!hs) {
        const __int128 c = (__int128)m_others * (m_others - 1) * (m_others - 2) / 6;
        if (c > (__int128)INT64_MAX / T) {
            set_error("simplicial counting: T*C(%lld,3) overflows int64 for T=%lld", (long long)m_others, (long long)T);
            return SD_ERR_OVERFLOW;
        }
    }
    // batch size: ~52 n bytes of keys and ranks per instance (+ the rank pipeline's part lists)
    i64 IB = (i64)((3ull << 30) / (size_t)(56 * n));
    if (IB < 1) IB = 1;
    if (IB > 32768) IB = 32768;
    if (IB > ninst_total) IB = ninst_total;
    SD_TRY(ctx->buf[BUF_IN2].reserve((size_t)IB * n * 3 * sizeof(double)));
    SD_TRY(ctx->buf[BUF_MASK].reserve((size_t)IB * n * 7 * sizeof(int)));
    double *KA = ctx->buf[BUF_IN2].as<double>();
    double *KB = KA + (size_t)IB * n;
    int *bA = ctx->buf[BUF_MASK].as<int>();
    int *aA = bA + (size_t)IB * n;
    int *bB = aA + (size_t)IB * n;
    int *aB = bB + (size_t)IB * 2 * n;
    int *claim = aB + (size_t)IB * 2 * n;
    ScGeom g;
    g.pts = d_pts;
    g.stride_j = stride_j;
    g.qidx = d_q;
    g.T = T;
    for (i64 i0 = 0; i0 < ninst_total; i0 += IB) {
        const i64 ni = ninst_total - i0 < IB ? ninst_total - i0 : IB;
        g.inst0 = i0;
        unsigned gx = (unsigned)ceil_div(n, 256 * 4);
        if (gx < 1) gx = 1;
        if (ni > 65535) {
            set_error("simplicial counting: internal batch too large");
            return SD_ERR_UNSUPPORTED;
        }
        sc_keys_kernel<<<dim3(gx, (unsigned)ni), 256, 0, st>>>(g, n, ni, tol, KA, KB, ctx->d_status);
        ctx->last.launches++;
        if (!hs) SD_CUDA(cudaMemsetAsync(claim, 0, (size_t)ni * n * sizeof(int), st));
        SD_TRY(rank_rows_device(ctx, KA, ni, n, n, bA, aA));
        SD_TRY(rank_rows_device(ctx, KB, ni, 2 * n, 2 * n, bB, tol > 0.0 || hs ? aB : nullptr));
        if (hs) hs_reduce_kernel<<<(unsigned)ni, 256, 0, st>>>(g, n, KA, KB, bA, aA, bB, aB, d_out, ctx->d_status);
        else if (tol > 0.0) sc_reduce_kernel<true><<<(unsigned)ni, 256, 0, st>>>(g, n, KA, KB, bA, aA, bB, aB, claim, m_others, d_out);
        else sc_reduce_kernel<false><<<(unsigned)ni, 256, 0, st>>>(g, n, KA, KB, bA, aA, bB, aB, claim, m_others, d_out);
        ctx->last.launches++;
        SD_CUDA(cudaGetLastError());
    }
    return SD_OK;
}


// ---------------------------------------------------------------------------------------------
// Oja depth, d = 2, in O(n log n) per query.  Replaces the enumeration of all pairs in _oja_depth
// (statdepth/depth/calculations/_pointcloud.py:176-204):  sum over pairs {a, b} of the pool of
// area(p, x_a, x_b) = |det(v_a, v_b)| / 2, v = x - p.  With the directions sorted by angle, every pair is
// counted once as (a, b) with b strictly inside the half-turn counter-clockwise of a, where det(v_a, v_b) > 0
// (pairs on one line through p have area 0), and det is linear in its second argument:
//     sum = 1/2 sum_a det(v_a, S_a),   S_a = sum of v_b over that half-turn
//         = prefix sums W[r] = sum of v_b with rank < r, taken at the rank of a's class end and of its antipode.
// Ranks come from the same two passes of the K1 pipeline as the triangle counting (exact keys, tolerance 0).
//
// Accuracy.  S_a is a difference of prefix sums of magnitude n |v|, and det(v_a, S_a) cancels when S_a is nearly
// parallel to v_a -- at every query far from the bulk, with float64 sums an error of n (R / spread) u.  So the sums
// are exact: every component of v is held in fixed point, c 2^(e-64) with 2^e above the query's largest component
// (from the pool's bounding box) and c = hi 2^32 + lo, hi in [-2^32, 2^32), lo in [0, 2^32]; the limbs add up in
// int64 without overflow for n < 2^30.  The only roundings left are c itself (2^(e-65), below the last bit of every
// component within 2^-11 of the largest), S_a to a pair of doubles (exact), det by fma-compensated products
// (u |det| + O(u^2) |v_a| |S_a|) and the sum of the non-negative dets (compensated per thread).
// Determinism.  Integer sums do not depend on their order, and the dets are added in a fixed order: the result
// is a function of the pool and the query alone (not of the call's other queries, their batch or the run).
// ---------------------------------------------------------------------------------------------
constexpr int OJ_THREADS = 512;

// bbox = {min x, max x, min y, max y} of the pool: with them fl(x_j - p) is bounded by the ends of the box
// (rounding is monotone), the largest component of every query's directions without a pass over the points.
__global__ void __launch_bounds__(1024) oja2_bbox_kernel(const double *__restrict__ pts, const i64 n,
                                                         double *__restrict__ bbox) {
    __shared__ double s[4][32];
    double lo[2] = {INFINITY, INFINITY}, hi[2] = {-INFINITY, -INFINITY};
    for (i64 j = threadIdx.x; j < n; j += blockDim.x)
#pragma unroll
        for (int c = 0; c < 2; ++c) {
            lo[c] = fmin(lo[c], pts[2 * j + c]);
            hi[c] = fmax(hi[c], pts[2 * j + c]);
        }
#pragma unroll
    for (int s2 = 16; s2 > 0; s2 >>= 1)
#pragma unroll
        for (int c = 0; c < 2; ++c) {
            lo[c] = fmin(lo[c], __shfl_xor_sync(0xffffffffu, lo[c], s2));
            hi[c] = fmax(hi[c], __shfl_xor_sync(0xffffffffu, hi[c], s2));
        }
    const int w = threadIdx.x >> 5, nw = blockDim.x >> 5;
    if ((threadIdx.x & 31) == 0) { s[0][w] = lo[0]; s[1][w] = hi[0]; s[2][w] = lo[1]; s[3][w] = hi[1]; }
    __syncthreads();
    if (threadIdx.x < 4) {
        double r = s[threadIdx.x][0];
        for (int k = 1; k < nw; ++k) r = threadIdx.x & 1 ? fmax(r, s[threadIdx.x][k]) : fmin(r, s[threadIdx.x][k]);
        bbox[threadIdx.x] = r;
    }
}

// v * 2^(64 - e) = hi 2^32 + lo (lo rounded to nearest), scale = 2^(32 - e), |v| < 2^e
__device__ __forceinline__ void oj_limbs(const double v, const double scale, u64 &hi, u64 &lo) {
    const double t = v * scale;  // exact: a power of two, |t| < 2^32
    const double f = floor(t);
    hi = (u64)(i64)f;
    lo = (u64)__double2ll_rn((t - f) * 4294967296.0);  // t - f in [0, 1) is exact
}

// the fixed-point value of limb sums (hi, lo) (two's complement, |value| < 2^93) as s + t exactly, times unit
__device__ __forceinline__ void oj_to_dd(const u64 hi, const u64 lo, const double unit, double &s, double &t) {
    const i64 h = (i64)(hi + (lo >> 32));
    const double hd = (double)h;                                       // |h - hd| <= 2^9
    const double a = hd * 4294967296.0;                                // exact
    const double b = (double)((h - (i64)hd) * 4294967296ll + (i64)(lo & 0xffffffffull));  // |.| < 2^42: exact
    s = a + b;                                                         // two-sum: s + t == a + b
    const double bb = s - a;
    t = (a - (s - bb)) + (b - bb);
    s *= unit;
    t *= unit;
}

// W[r] = {hi x, lo x, hi y, lo y} limb sums: exclusive prefix over ranks after pass 2
struct OjW { u64 hx, lx, hy, ly; };
__device__ __forceinline__ OjW oj_load(const u64 *w, const i64 r) {
    const ulonglong2 a = reinterpret_cast<const ulonglong2 *>(w + 4 * r)[0];
    const ulonglong2 b = reinterpret_cast<const ulonglong2 *>(w + 4 * r)[1];
    return OjW{a.x, a.y, b.x, b.y};
}

__global__ void __launch_bounds__(OJ_THREADS) oja2_reduce_kernel(const ScGeom g, const i64 n, const double *__restrict__ KA,
                                                                 const int *__restrict__ bA, const int *__restrict__ aA,
                                                                 const int *__restrict__ bB, u64 *__restrict__ bucket,
                                                                 const double *__restrict__ bbox,
                                                                 const double hull_volume, double *__restrict__ out) {
    __shared__ u64 s_part[4][OJ_THREADS];
    __shared__ double s_red[OJ_THREADS / 32];
    __shared__ i64 s_cnt[2];
    const i64 li = blockIdx.x;
    const i64 inst = g.inst0 + li;
    const i64 q = sc_query(g, inst);
    const double px = g.pts[q * g.stride_j], py = g.pts[q * g.stride_j + 1];
    const double *ka = KA + li * n;
    const int *ba = bA + li * n, *aa = aA + li * n, *bb = bB + li * 2 * n;
    u64 *W = bucket + li * 4 * (n + 1);
    const int tid = threadIdx.x;
    // the fixed-point scale of this query: 2^e > every |component| of its directions
    const double M = fmax(fmax(fabs(bbox[0] - px), fabs(bbox[1] - px)), fmax(fabs(bbox[2] - py), fabs(bbox[3] - py)));
    int e;
    frexp(M, &e);  // M < 2^e (M == 0: every direction is zero, e = 0)
    const double scale = ldexp(1.0, 32 - e), unit = ldexp(1.0, e - 64);
    for (i64 r = tid; r < 2 * (n + 1); r += OJ_THREADS) reinterpret_cast<ulonglong2 *>(W)[r] = make_ulonglong2(0, 0);
    if (tid == 0) { s_cnt[0] = 0; s_cnt[1] = 0; }
    __syncthreads();
    // pass 1: limb sums by rank, #real directions and #directions in [0, pi)
    i64 real = 0, low = 0;
    for (i64 j = tid; j < n; j += OJ_THREADS) {
        const double u = ka[j];
        if (!(u < 16.0)) continue;
        u64 hx, lx, hy, ly;
        oj_limbs(g.pts[j * g.stride_j] - px, scale, hx, lx);
        oj_limbs(g.pts[j * g.stride_j + 1] - py, scale, hy, ly);
        u64 *w = W + 4 * (i64)ba[j];
        atomicAdd(w, hx);
        atomicAdd(w + 1, lx);
        atomicAdd(w + 2, hy);
        atomicAdd(w + 3, ly);
        ++real;
        low += u < 12.0;
    }
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) {
        real += __shfl_xor_sync(0xffffffffu, real, s);
        low += __shfl_xor_sync(0xffffffffu, low, s);
    }
    if ((tid & 31) == 0) {
        atomicAdd((u64 *)&s_cnt[0], (u64)real);
        atomicAdd((u64 *)&s_cnt[1], (u64)low);
    }
    __syncthreads();
    // pass 2: exclusive scan of the limb sums in place: W[r] = sum of v_b with rank < r   (r = 0 .. n; W[n] = total)
    const i64 len = n + 1, chunk = (len + OJ_THREADS - 1) / OJ_THREADS;
    const i64 c0 = tid * chunk, c1 = c0 + chunk < len ? c0 + chunk : len;
    u64 acc4[4] = {0, 0, 0, 0};
    for (i64 r = c0; r < c1; ++r) {
        const OjW v = oj_load(W, r);
        acc4[0] += v.hx; acc4[1] += v.lx; acc4[2] += v.hy; acc4[3] += v.ly;
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) s_part[k][tid] = acc4[k];
    __syncthreads();
    if (tid < 4) {  // 512 partial sums per limb: a serial scan by one thread each is negligible
        u64 run = 0;
        for (int k = 0; k < OJ_THREADS; ++k) { const u64 v = s_part[tid][k]; s_part[tid][k] = run; run += v; }
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 4; ++k) acc4[k] = s_part[k][tid];
    for (i64 r = c0; r < c1; ++r) {
        const OjW v = oj_load(W, r);
        reinterpret_cast<ulonglong2 *>(W + 4 * r)[0] = make_ulonglong2(acc4[0], acc4[1]);
        reinterpret_cast<ulonglong2 *>(W + 4 * r)[1] = make_ulonglong2(acc4[2], acc4[3]);
        acc4[0] += v.hx; acc4[1] += v.lx; acc4[2] += v.hy; acc4[3] += v.ly;
    }
    __syncthreads();
    // pass 3: det(v_a, S_a) from the exact half-turn sums
    const i64 mreal = s_cnt[0], L4 = s_cnt[1], H = mreal - L4;
    const OjW tot = oj_load(W, n);
    double acc = 0.0, comp = 0.0;
    for (i64 j = tid; j < n; j += OJ_THREADS) {
        const double u = ka[j];
        if (!(u < 16.0)) continue;
        const double vx = g.pts[j * g.stride_j] - px, vy = g.pts[j * g.stride_j + 1] - py;
        const i64 L = ba[j], R = n - (i64)aa[j];  // ranks [L, R) hold the class of j
        const i64 b2w = bb[n + j];
        const OjW wr = oj_load(W, R);
        OjW S;
        if (u < 12.0) {
            const OjW ww = oj_load(W, b2w - L - H);  // real directions strictly before the antipode
            S = OjW{ww.hx - wr.hx, ww.lx - wr.lx, ww.hy - wr.hy, ww.ly - wr.ly};
        } else {
            const OjW ww = oj_load(W, b2w - L + L4);
            S = OjW{tot.hx - wr.hx + ww.hx, tot.lx - wr.lx + ww.lx, tot.hy - wr.hy + ww.hy, tot.ly - wr.ly + ww.ly};
        }
        double sx, tx, sy, ty;
        oj_to_dd(S.hx, S.lx, unit, sx, tx);
        oj_to_dd(S.hy, S.ly, unit, sy, ty);
        const double p1 = vx * sy, e1 = fma(vx, sy, -p1);
        const double p2 = vy * sx, e2 = fma(vy, sx, -p2);
        const double d = (p1 - p2) + ((e1 - e2) + (vx * ty - vy * tx));
        const double t = acc + d;  // two-sum
        const double z = t - acc;
        comp += (acc - (t - z)) + (d - z);
        acc = t;
    }
    acc += comp;
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, s);
    if ((tid & 31) == 0) s_red[tid >> 5] = acc;
    __syncthreads();
    if (tid == 0) {
        double sum = 0.0;
        for (int w = 0; w < OJ_THREADS / 32; ++w) sum += s_red[w];
        out[inst] = 0.5 * sum / hull_volume;
    }
}

// d_pts: the pool's points [n][2] (already gathered); d_q: positions of the queries inside the pool
int oja2_count_device(sd_ctx *ctx, const double *d_pts, i64 n, const i64 *d_q, i64 nq, double hull_volume,
                      double *d_out) {
    cudaStream_t st = ctx->stream;
    if (nq == 0) return SD_OK;
    if (n < 3) {  // no pair of other points
        SD_CUDA(cudaMemsetAsync(d_out, 0, (size_t)nq * sizeof(double), st));
        return SD_OK;
    }
    if (2 * n >= (1ll << 31)) {
        set_error("oja counting: n=%lld too large", (long long)n);
        return SD_ERR_UNSUPPORTED;
    }
    // batch size: ~88 n bytes of keys, limb sums and ranks per query (+ the rank pipeline's part lists)
    i64 IB = (i64)((3ull << 30) / (size_t)(88 * n));
    if (IB < 1) IB = 1;
    if (IB > 32768) IB = 32768;
    if (IB > nq) IB = nq;
    SD_TRY(ctx->buf[BUF_IN2].reserve((size_t)IB * (3 * n + 4 * (n + 1)) * sizeof(double) + 4 * sizeof(double)));
    SD_TRY(ctx->buf[BUF_MASK].reserve((size_t)IB * n * 4 * sizeof(int)));
    u64 *bucket = ctx->buf[BUF_IN2].as<u64>();  // first: 16-byte loads and stores, 32 (n + 1) bytes per query
    double *KA = reinterpret_cast<double *>(bucket + (size_t)IB * 4 * (n + 1));
    double *KB = KA + (size_t)IB * n;
    double *bbox = KB + (size_t)IB * 2 * n;
    int *bA = ctx->buf[BUF_MASK].as<int>();
    int *aA = bA + (size_t)IB * n;
    int *bB = aA + (size_t)IB * n;
    ScGeom g;
    g.pts = d_pts;
    g.stride_j = 2;
    g.qidx = d_q;
    g.T = 1;
    oja2_bbox_kernel<<<1, 1024, 0, st>>>(d_pts, n, bbox);
    ctx->last.launches++;
    for (i64 i0 = 0; i0 < nq; i0 += IB) {
        const i64 ni = nq - i0 < IB ? nq - i0 : IB;
        g.inst0 = i0;
        unsigned gx = (unsigned)ceil_div(n, 256 * 4);
        if (gx < 1) gx = 1;
        sc_keys_kernel<<<dim3(gx, (unsigned)ni), 256, 0, st>>>(g, n, ni, 0.0, KA, KB, ctx->d_status);
        ctx->last.launches++;
        SD_TRY(rank_rows_device(ctx, KA, ni, n, n, bA, aA));
        SD_TRY(rank_rows_device(ctx, KB, ni, 2 * n, 2 * n, bB, nullptr));
        oja2_reduce_kernel<<<(unsigned)ni, OJ_THREADS, 0, st>>>(g, n, KA, bA, aA, bB, bucket, bbox, hull_volume, d_out);
        ctx->last.launches++;
        SD_CUDA(cudaGetLastError());
    }
    return SD_OK;
}

}  // namespace sd
