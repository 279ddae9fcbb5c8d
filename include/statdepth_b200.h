/*
 * statdepth_b200.h -- C ABI of the B200-native depth engine (libsdepth.so).
 *
 * Drop-in boundary for statdepth's data-parallel hot path.  The reference has no FFI: its seam is
 * two private Python drivers imported by name in statdepth/depth/depth.py:7-8,
 *     _functionaldepth(data, to_compute, J, containment, relax, deep_check, quiet) -> pd.Series
 *         (statdepth/depth/calculations/_functional.py:17-97)
 *     _pointwisedepth(data, to_compute, containment, quiet) -> pd.Series
 *         (statdepth/depth/calculations/_pointcloud.py:14-66)
 * Each entry point below replaces the inner loops of one of those drivers and returns the
 * INTEGER numerators (or float64 depths where the reference's result is a float sum); the Python
 * host (statdepth_b200/) turns them into the same pd.Series the reference returns.  The ctypes
 * binding a maintainer of the reference would add is shown in INTEGRATION.md.
 *
 * Conventions
 *   - plain pointers and sizes only; the caller owns every host buffer, the library owns all
 *     device memory (per-context workspace, grown on demand, freed by sd_destroy);
 *   - every function returns an int status (SD_OK == 0), never throws or aborts;
 *     sd_last_error() returns a thread-local, NUL-terminated description of the last failure;
 *   - every call is synchronous on return; internally stream-ordered on the context's stream;
 *   - one context per GPU per process (one process per GPU; multi-GPU sharding is done by the
 *     host with torch.distributed, see DESIGN.md "Multi-GPU");
 *   - `*_dev` variants take DEVICE pointers (e.g. torch tensors' data_ptr()) and do no copies:
 *     they are what bench.py times as the HBM-resident `value`.
 *   - non-finite inputs are rejected with SD_ERR_NONFINITE (documented divergence: the reference
 *     silently skips NaNs through pandas min/max, _containment.py:68-69).
 */
#ifndef STATDEPTH_B200_H
#define STATDEPTH_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SD_ABI_VERSION 1

typedef struct sd_ctx sd_ctx;

enum sd_status {
    SD_OK = 0,
    SD_ERR_INVALID = 1,     /* bad argument (null pointer, negative size, unsupported J/d/layout) */
    SD_ERR_CUDA = 2,        /* a CUDA runtime call failed; text in sd_last_error() */
    SD_ERR_NO_DEVICE = 3,   /* no usable sm_100 device */
    SD_ERR_NONFINITE = 4,   /* NaN or +-inf in the input */
    SD_ERR_OVERFLOW = 5,    /* integer numerator would exceed int64 for this (n, T, J); a squared distance overflows */
    SD_ERR_UNSUPPORTED = 6  /* configuration the engine does not implement (no CPU fallback) */
};

/* layout of the univariate matrix handed to sd_band_depth_f64 */
enum sd_layout {
    SD_LAYOUT_TN = 0, /* X[t*ld + c]: T time rows, n curves, ld >= n  (== DataFrame.to_numpy(), C order) */
    SD_LAYOUT_NT = 1  /* X[c*ld + t]: n curve rows, T points, ld >= T (== F-ordered DataFrame values)   */
};

/* strict band-depth kernel selection (sd_set_option(ctx, SD_OPT_BD_IMPL, ...)) */
enum sd_bd_impl {
    SD_BD_AUTO = 0,  /* sign-vector matching when it applies; queries it cannot certify (ties with the query,
                        n > 8193) go to the bit kernel, or to the dense Gram if a probe of 8 queries shows that
                        more than 2 % of all pairs survive the first mask word */
    SD_BD_BITS = 1,  /* bit-packed AND + early exit on CUDA cores                      */
    SD_BD_GEMM = 2,  /* int8 violation Gram V = Sb Sb^T + Sa Sa^T on tcgen05 / TMEM    */
    SD_BD_MATCH = 3  /* complementary sign-vector matching (O(nT) per query) + enumeration of uncertified queries */
};

enum sd_option {
    SD_OPT_BD_IMPL = 1,       /* enum sd_bd_impl */
    SD_OPT_MBD_FORCE_FALLBACK = 2, /* 1: rank every row with the generic (slow) path; testing aid */
    SD_OPT_PROFILE = 3,           /* 1: bracket every kernel phase with CUDA events (sd_get_phase_ns) */
    SD_OPT_SIMPLICIAL_IMPL = 4,   /* enum sd_simplicial_impl: 2-D triangle counting algorithm */
    SD_OPT_ASYNC_DEVICE = 5       /* 1: sd_band_depth_f64_dev (relax = 1) only ENQUEUES its work on sd_stream() and
                                     returns; status, timings and the result are valid after sd_sync().  Lets a caller
                                     queue a collective behind the kernels without a host round trip. */
};

/* how 2-D simplicial counts (point clouds, relaxed multivariate simplex depth) are obtained */
enum sd_simplicial_impl {
    SD_SIMPLICIAL_AUTO = 0,      /* enumerate samples of up to 64 points / curves, count larger ones (d = 2); same semantics */
    SD_SIMPLICIAL_ENUMERATE = 1, /* all (d+1)-subsets, closed simplex test with tolerance `tol` */
    SD_SIMPLICIAL_COUNT = 2      /* O(n log n) angular counting, d = 2: dist(p, triangle) <= tol; tol = 0: exact closed triangles */
};

/* phases of the modified-band-depth pipeline reported by sd_get_phase_ns */
enum sd_phase {
    SD_PHASE_MBD_SPLITTERS = 0,
    SD_PHASE_MBD_PARTITION = 1,
    SD_PHASE_MBD_RANK = 2,
    SD_PHASE_MBD_GENERIC = 3,
    SD_PHASE_BD_MASKS = 4,
    SD_PHASE_BD_PAIRS = 5,
    SD_PHASE_MBD_SLAB_HIST = 6, /* slab path: table + hist kernels (range, code table, per-value codes, bin starts) */
    SD_PHASE_MBD_SLAB_RANK = 7, /* slab path: rank kernel */
    SD_PHASE_COUNT = 8
};

/* nanoseconds of the LAST call on this context, from CUDA events on the context's stream */
typedef struct sd_timings {
    int64_t h2d_ns;      /* host->device copies                */
    int64_t kernel_ns;   /* all kernels of the call            */
    int64_t d2h_ns;      /* device->host copy of the result    */
    int64_t launches;    /* number of kernel launches          */
    int64_t fallback_rows; /* MBD: time rows ranked by the generic path (0 on well-spread data) */
    int64_t bd_impl_used;  /* strict band depth: enum sd_bd_impl that did (most of) the work, 0 if n/a */
} sd_timings;

typedef struct sd_devinfo {
    int device;
    int sm_count;
    int cc_major, cc_minor;
    int64_t total_mem;
    char name[128];
} sd_devinfo;

int sd_abi_version(void);
const char *sd_last_error(void);

/* create / destroy a context on CUDA device `device` (creates a stream and timing events). */
int sd_init(int device, sd_ctx **out);
int sd_destroy(sd_ctx *ctx);
int sd_device_info(sd_ctx *ctx, sd_devinfo *out);
int sd_set_option(sd_ctx *ctx, int option, int64_t value);
int sd_get_timings(sd_ctx *ctx, sd_timings *out);
/* with SD_OPT_PROFILE on: device nanoseconds per phase (enum sd_phase) of the LAST call, summed over
 * its launches of that phase; out must hold SD_PHASE_COUNT entries. */
int sd_get_phase_ns(sd_ctx *ctx, int64_t *out);
/* micro-benchmark: sustained tcgen05.mma kind::i8 rate of this GPU in int8 ops/s (2 per MAC), the measured
 * denominator for the Gram kernel's roofline fraction (takes ~10 ms) */
int sd_probe_int8_peak(sd_ctx *ctx, double *ops_per_s);
/* the context's cudaStream_t (as void*), so a caller can order its own work / events on it */
void *sd_stream(sd_ctx *ctx);
/* waits for everything queued on sd_stream(); with SD_OPT_ASYNC_DEVICE it completes the pending
 * sd_band_depth_f64_dev call (returns its status, makes sd_get_timings valid) */
int sd_sync(sd_ctx *ctx);
/* Which rank pipeline relaxed depth takes for rows of n curves with leading dimension ld, and its geometry (host
 * arithmetic only: no context, no GPU).  out6[0] = 1: slab path (csrc/mbd_slab.cuh), 0: part pipeline; for the slab
 * path out6[1] = rank CTAs per row, [2] = bins per CTA, [3] = entries one CTA may hold, [4] / [5] = dynamic shared
 * memory of the rank / hist kernel in bytes.  The device pointer is assumed 16-byte aligned; the SD_MBD_* environment
 * variables apply as they do to the depth calls. */
int sd_mbd_plan(int64_t n, int64_t ld, int64_t *out6);

/*
 * Univariate band depth numerators.  Replaces _univariate_band_depth (_functional.py:198-255)
 * + _r2_containment (_containment.py:45-80) + _subsequences (_helper.py:16-32) for one j.
 *
 *   relax == 0 : count_out[q] = #{j-subsets S of the other n-1 curves : the band of S contains
 *                curve query_idx[q] at ALL T points}              (closed interval, J = 2 or 3)
 *   relax != 0 : count_out[q] = sum_t #{j-subsets whose band contains the curve at time t}
 *                             = sum_t [C(n-1,j) - C(b_t,j) - C(a_t,j)]
 * The host forms  depth = sum_{j=2..J} count_j [/ T] / C(n, j)   (_functional.py:229,253).
 *
 * query_idx == NULL means all n curves (nq must then equal n).  T-sharding for multi-GPU MBD:
 * pass a block of time rows; relaxed counts are additive over disjoint row blocks.
 */
int sd_band_depth_f64(sd_ctx *ctx, const double *X, int64_t T, int64_t n, int64_t ld, int layout,
                      const int64_t *query_idx, int64_t nq, int j, int relax, int64_t *count_out);

/* same, X / query_idx / count_out are DEVICE pointers, layout SD_LAYOUT_TN only */
int sd_band_depth_f64_dev(sd_ctx *ctx, const double *dX, int64_t T, int64_t n, int64_t ld,
                          const int64_t *d_query_idx, int64_t nq, int j, int relax,
                          int64_t *d_count_out);

/*
 * Per-(time, curve) strict ranks: below[t*n + c] = #curves strictly below curve c at time t,
 * above[...] likewise (int32).  The integer intermediates SURVEY 8a calls "rank/count
 * intermediates"; also what relaxed depth for J >= 4 is assembled from on the host.
 */
int sd_band_ranks_f64(sd_ctx *ctx, const double *X, int64_t T, int64_t n, int64_t ld, int layout,
                      int32_t *below_out, int32_t *above_out);

/*
 * Multivariate functional simplex depth numerators.  Replaces _simplex_depth
 * (_functional.py:257-286) + _simplex_containment / _is_in_simplex (_containment.py:105-176).
 * F[(i*T + t)*d + c]: N curves, T rows, d in {1,2,3} channels.  tol = absolute tolerance band
 * of the closed simplex test (the reference's LP accepts ~1e-7; pass 0 for exact sign tests).
 *   relax == 0 : #{(d+1)-subsets of the other N-1 curves containing the query at all T rows}
 *   relax != 0 : sum over subsets of #rows contained
 * SD_ERR_OVERFLOW when relax != 0, d = 2, the counts are counted (enum sd_simplicial_impl) and T * C(N-1, 3)
 * exceeds int64 (T = 1: N > 3 810 780; T = 64: N > 952 696).
 */
int sd_simplex_depth_f64(sd_ctx *ctx, const double *F, int64_t N, int64_t T, int d,
                         const int64_t *query_idx, int64_t nq, int relax, double tol,
                         int64_t *count_out);

/* Point cloud P[i*d + c], n points.  Replaces the 'simplex' branch of _pointwisedepth
 * (_pointcloud.py:44-56): #{(d+1)-subsets of the other points whose closed simplex contains p}.
 * SD_ERR_OVERFLOW when d = 2, the counts are counted (enum sd_simplicial_impl) and C(n-1, 3) exceeds int64
 * (n > 3 810 780). */
int sd_pointcloud_simplicial_f64(sd_ctx *ctx, const double *P, int64_t n, int d,
                                 const int64_t *query_idx, int64_t nq, double tol,
                                 int64_t *count_out);

/* Replaces _L1_depth (_pointcloud.py:125-150): 1 - ||sum_{o!=p} (x_o-x_p)/||x_p-x_o|| || / n. */
int sd_pointcloud_l1_f64(sd_ctx *ctx, const double *P, int64_t n, int d, const int64_t *query_idx,
                         int64_t nq, double *depth_out);

/* Replaces _oja_depth (_pointcloud.py:176-204): sum over d-subsets S of pool\{p} of
 * vol(conv(S u {p})) / hull_volume.  pool == NULL means all n points. */
int sd_pointcloud_oja_f64(sd_ctx *ctx, const double *P, int64_t n, int d, const int64_t *query_idx,
                          int64_t nq, const int64_t *pool, int64_t npool, double hull_volume,
                          double *out);

/*
 * B small sub-clouds of one cloud with ONE query each, in one launch: what K-sampled point-cloud depth consists
 * of (_samplepointwisedepth, _pointcloud.py:97-123).  Block b holds the points member[block_off[b] .. block_off[b+1])
 * (ids into P, in the reference's order: the L1 sum runs in that order, bit for bit), its query is the member at
 * position query_pos[b].  kind 0: simplicial count (returned as a double, exact below 2^53), 1: L1 depth,
 * 2: Oja sum / hull_volume[b] (d in {2,3}).  At most 4096 / d members per block (they are enumerated).
 */
int sd_pointcloud_blocks_f64(sd_ctx *ctx, const double *P, int64_t n, int d, const int64_t *member,
                             const int64_t *block_off, const int64_t *query_pos, int64_t B, int kind, double tol,
                             const double *hull_volume, double *out);

/*
 * Out-of-sample depth: the depth of NEW observations Y against a reference sample S.  The value for new
 * observation g is what the in-sample entry point returns for g after g alone is appended to S (the reference:
 * FunctionalDepth([pd.concat([S, g], axis=1)], to_compute=[g]) / PointcloudDepth(pd.concat([S, g]), ...)).
 * Other new observations never take part in g's depth.  The host forms the depth with the population size
 * nS + 1, e.g. relaxed band depth = sum_j count_j / T / C(nS + 1, j).
 *
 * Band depth, S [T, nS] and Y [T, nY] in SD_LAYOUT_TN (S[t*ldS + c], Y[t*ldY + g]), j = 2 or 3:
 *   relax != 0 : count_out[g] = sum_t [C(nS,j) - C(b_t,j) - C(a_t,j)], b_t / a_t = #sample curves strictly
 *                below / above Y[t, g].  O((nS + nY) T): two exact rank passes (pooled [S | Y], and Y alone),
 *                b_t = below among the pool - below among Y.
 *   relax == 0 : count_out[g] = #{j-subsets of the nS sample curves whose band contains curve g at all T
 *                points}.  Always the bit-mask kernels (SD_BD_BITS): the sign-vector matcher and the Gram
 *                route are not used here, so tie-heavy strict data costs what the bit kernel costs.
 * SD_ERR_OVERFLOW when T * C(nS, j) exceeds int64.
 */
int sd_band_depth_oos_f64(sd_ctx *ctx, const double *S, int64_t T, int64_t nS, int64_t ldS,
                          const double *Y, int64_t nY, int64_t ldY, int j, int relax,
                          int64_t *count_out);

/* same with DEVICE pointers (count_out too).  When Y is the continuation of S in one matrix
 * (dY == dS + nS, ldY == ldS) the data is used in place; otherwise it is first pooled on the device. */
int sd_band_depth_oos_f64_dev(sd_ctx *ctx, const double *dS, int64_t T, int64_t nS, int64_t ldS,
                              const double *dY, int64_t nY, int64_t ldY, int j, int relax,
                              int64_t *d_count_out);

/*
 * A fitted reference: the same relaxed counts from the sample's sorted rows, so that a sample scored against again
 * and again is sorted once and only the new curves cross to the device on each call.
 *
 * Sorted reference rows (the index of a fitted reference): d_sorted_out[t*nS + k] = the k-th smallest of
 * dX[t*ld + 0 .. nS), ties repeated.  Device pointers, SD_LAYOUT_TN, d_sorted_out holds T*nS doubles.
 * SD_ERR_NONFINITE when the sample holds NaN or +-inf.
 */
int sd_band_sort_rows_f64_dev(sd_ctx *ctx, const double *dX, int64_t T, int64_t nS, int64_t ld,
                              double *d_sorted_out);

/* Relaxed out-of-sample band depth numerators from sorted rows, J = 2 or 3:
 * d_count_out[(j-2)*nY + g] = sum_t [C(nS,j) - C(b_t,j) - C(a_t,j)], j = 2..J, b_t / a_t = #values of sorted row t
 * strictly below / above dY[t*ldY + g] -- equal to sd_band_depth_oos_f64_dev(relax = 1, j).  Device pointers,
 * d_count_out holds (J - 1)*nY int64.  SD_ERR_NONFINITE when Y holds NaN or +-inf, SD_ERR_OVERFLOW when
 * T * C(nS, J) exceeds int64. */
int sd_band_depth_sorted_f64_dev(sd_ctx *ctx, const double *d_sorted, int64_t T, int64_t nS,
                                 const double *dY, int64_t nY, int64_t ldY, int J, int64_t *d_count_out);

/* Point clouds S[i*d + c] (nS points) and Y[g*d + c] (nY points), d in 1..3:
 * count_out[g] = #{(d+1)-subsets of S whose closed simplex contains Y[g]} with the tolerance band `tol` of
 * sd_pointcloud_simplicial_f64 (enumerated, or counted for d = 2 when nS + 1 > 64, as there).
 * The host divides by C(nS + 1, d + 1).  SD_ERR_OVERFLOW when d = 2, the counts are counted and C(nS, 3) exceeds
 * int64 (nS > 3 810 779). */
int sd_pointcloud_simplicial_oos_f64(sd_ctx *ctx, const double *S, int64_t nS, int d,
                                     const double *Y, int64_t nY, double tol, int64_t *count_out);

/* depth_out[g] = 1 - ||sum_{s in S} (s - y)/||s - y|| || / (nS + 1), d in 1..16 (NaN when y equals a
 * sample point, as in the reference). */
int sd_pointcloud_l1_oos_f64(sd_ctx *ctx, const double *S, int64_t nS, int d, const double *Y,
                             int64_t nY, double *depth_out);

/*
 * Functional outlier detection (functional boxplot, outliergram).  X [T, n] in `layout`, as sd_band_depth_f64.
 *
 * Rank sums.  With b_t(c) / a_t(c) the number of OTHER curves strictly below / above curve c at row t:
 *   q_out[c]         = sum_t [C(n-1,2) - C(b_t,2) - C(a_t,2)]   (== sd_band_depth_f64(relax = 1, j = 2))
 *   below_sum_out[c] = sum_t b_t,   above_sum_out[c] = sum_t a_t  (above_sum_out may be NULL)
 * exact int64; SD_ERR_OVERFLOW when T * C(n-1, 2) exceeds int64.  All three are additive over disjoint blocks of
 * time rows.  The modified epigraph index of the outliergram is 1 - below_sum / (n T).
 */
int sd_band_rank_sums_f64(sd_ctx *ctx, const double *X, int64_t T, int64_t n, int64_t ld, int layout,
                          int64_t *q_out, int64_t *below_sum_out, int64_t *above_sum_out);

/* same with DEVICE pointers, SD_LAYOUT_TN only */
int sd_band_rank_sums_f64_dev(sd_ctx *ctx, const double *dX, int64_t T, int64_t n, int64_t ld,
                              int64_t *d_q_out, int64_t *d_below_sum_out, int64_t *d_above_sum_out);

/*
 * Masked envelope.  member[c] != 0 selects the curves the envelope is taken over (SD_ERR_INVALID if it selects
 * none).  Per row t: lower_out[t] / upper_out[t] = min / max of X[t, c] over the member curves.
 * outside_out[c] (may be NULL) = #rows t with X[t, c] < lo_t - f or X[t, c] > hi_t + f, f = factor * (hi_t - lo_t)
 * (factor finite and >= 0); each of the four operations is one correctly rounded double operation (no fused
 * multiply-add), so a caller rebuilds the same fences from lower_out / upper_out.  A value on a fence is not
 * outside.  Rows are independent: a block of time rows gives those rows' envelope and its share of outside_out,
 * which is additive over disjoint row blocks.
 */
int sd_band_envelope_f64(sd_ctx *ctx, const double *X, int64_t T, int64_t n, int64_t ld, int layout,
                         const uint8_t *member, double factor, double *lower_out, double *upper_out,
                         int64_t *outside_out);

/* same with DEVICE pointers (member and outputs too), SD_LAYOUT_TN only */
int sd_band_envelope_f64_dev(sd_ctx *ctx, const double *dX, int64_t T, int64_t n, int64_t ld,
                             const uint8_t *d_member, double factor, double *d_lower_out, double *d_upper_out,
                             int64_t *d_outside_out);

/*
 * Extremal depth (Narisetty & Nair 2016).  b_t(c) / a_t(c) as for the rank sums above.
 *
 * Pointwise extremity: d_m_out[t*n + c] = |b_t(c) - a_t(c)| in [0, n - 1] (int32, row-major; the paper's pointwise
 * depth is 1 - m / n).  Device pointers, SD_LAYOUT_TN.  Rows are independent: a block of time rows gives those rows
 * of m.  SD_ERR_NONFINITE when X holds NaN or +-inf.
 */
int sd_band_extremity_f64_dev(sd_ctx *ctx, const double *dX, int64_t T, int64_t n, int64_t ld, int32_t *d_m_out);

/* Numerators from the full extremity matrix d_m [T, n] (row-major): with key(c) = (m_t(c))_t sorted descending and
 * keys compared lexicographically (larger = more extreme), d_num_out[c] = #{h : key(h) >= key(c)} in [1, n];
 * ED = d_num_out / n, equal keys get equal numerators.  Device pointers, d_num_out holds n int64.  SD_ERR_INVALID
 * when an m value lies outside [0, n - 1], when n > INT32_MAX, or when T > SD_EXTREMAL_T_MAX. */
#define SD_EXTREMAL_T_MAX 16384
int sd_extremal_depth_dev(sd_ctx *ctx, const int32_t *d_m, int64_t T, int64_t n, int64_t *d_num_out);

/*
 * Halfspace (Tukey) depth numerators, exact int64 (decisions: exact angular keys, no tolerance band).
 * h(p) = min over closed half-planes H whose boundary passes through p of #{i : x_i in H}, p itself counted; the host
 * divides by n.  d = 1: h = n - max(b, a), b / a the other points strictly below / above p.  d = 2: with z = #points
 * equal to p (p included), the m directions v_i = x_i - p != 0 and k_i = #{directions in the half-turn
 * (phi_i, phi_i + pi]}, h = z + min_i min(k_i, m - k_i), and h = n when m = 0.  Directions are compared by the exact
 * angular keys of the computed float64 differences (the tol = 0 decisions of the simplicial counting).
 * SD_ERR_NONFINITE when the input holds NaN or +-inf; SD_ERR_UNSUPPORTED for another d, and beyond the size limits
 * of the angular counting (2n < 2^31, d = 2) and of the rank pipeline (n < 2^31).
 */
int sd_pointcloud_halfspace_f64(sd_ctx *ctx, const double *P, int64_t n, int d, const int64_t *query_idx,
                                int64_t nq, int64_t *count_out);             /* d in {1,2}; count in [1, n] */
int sd_functional_halfspace_f64(sd_ctx *ctx, const double *F, int64_t N, int64_t T, int d,
                                const int64_t *query_idx, int64_t nq, int64_t *count_out);
                                /* F[(i*T + t)*d + c] as sd_simplex_depth_f64, d = 2; sum_t h_t in [T, T*N] */
int sd_band_halfspace_f64(sd_ctx *ctx, const double *X, int64_t T, int64_t n, int64_t ld, int layout,
                          int64_t *count_out);                               /* univariate, all n curves */

/* same with DEVICE pointers, SD_LAYOUT_TN only; additive over disjoint blocks of time rows */
int sd_band_halfspace_f64_dev(sd_ctx *ctx, const double *dX, int64_t T, int64_t n, int64_t ld,
                              int64_t *d_count_out);

/*
 * Random projection depths of curves F [N, T, d] (F[(i*T + t)*d + c] as sd_simplex_depth_f64; a point cloud is
 * T = 1) along K directions U [K, d] (row-major, used as given: rows must be finite and non-zero; U is HOST memory
 * in every variant, checked before it is uploaded).  Each (t, k) gives N projections
 *     y_k(i, t) = (...((U[k,0] F[i,t,0]) + U[k,1] F[i,t,1]) + ...) + U[k,d-1] F[i,t,d-1]
 * summed in this order with correctly rounded products and sums (no FMA, no tensor cores).
 *
 * Random Tukey depth: count_out[i] = sum_t min_k (N - max(b, a)) in [T, T*N], b / a the other projections of the
 * row strictly below / above; depth = count / (T N).  Equal to the exact halfspace depth numerator when U holds a
 * direction inside every cell of the arrangement, an upper bound on it otherwise.
 * Projection outlyingness: o_out[t*N + i] = max_k |y - med| / MAD with med = np.median of the row and the unscaled
 * MAD = np.median(|y - med|); MAD = 0 gives 0 where y == med and +inf elsewhere.  med_out / mad_out [T, K]
 * (t-major) may be NULL.  Projection depth is 1 / (1 + O).
 *
 * SD_ERR_INVALID for N, T, d or K < 1 and for a zero or non-finite direction row; SD_ERR_NONFINITE when F holds NaN
 * or +-inf or a projection overflows; SD_ERR_UNSUPPORTED for N >= 2^31.
 */
int sd_projection_tukey_f64(sd_ctx *ctx, const double *F, int64_t N, int64_t T, int d, const double *U, int64_t K,
                            int64_t *count_out);
int sd_projection_outlyingness_f64(sd_ctx *ctx, const double *F, int64_t N, int64_t T, int d, const double *U,
                                   int64_t K, double *o_out, double *med_out, double *mad_out);
/* univariate curves X [T, n] in either layout: the single direction u = 1 (y = x), o_out [T, n], med / mad [T] */
int sd_band_outlyingness_f64(sd_ctx *ctx, const double *X, int64_t T, int64_t n, int64_t ld, int layout,
                             double *o_out, double *med_out, double *mad_out);

/* same with DEVICE pointers for F / X and the outputs (U stays host memory); SD_LAYOUT_TN only */
int sd_projection_tukey_f64_dev(sd_ctx *ctx, const double *dF, int64_t N, int64_t T, int d, const double *U,
                                int64_t K, int64_t *d_count_out);
int sd_projection_outlyingness_f64_dev(sd_ctx *ctx, const double *dF, int64_t N, int64_t T, int d,
                                       const double *U, int64_t K, double *d_o_out, double *d_med_out,
                                       double *d_mad_out);
int sd_band_outlyingness_f64_dev(sd_ctx *ctx, const double *dX, int64_t T, int64_t n, int64_t ld, double *d_o_out,
                                 double *d_med_out, double *d_mad_out);

/*
 * Fitted references for random projection depths: the depth of NEW observations against a reference sample S, with
 * the out-of-sample convention above (new observation g gets what the in-sample entry point returns for g after g
 * alone is appended to S, with the same directions).  The reference's projections are sorted once; each query reads
 * only the new observations and binary-searches them in the sorted rows.
 *
 * Index: d_sorted_out[(t*K + k)*nS + j] = the j-th smallest of the projections y_k(i, t) of the nS curves dF [nS, T, d]
 * (as sd_projection_*: a point cloud is T = 1, U host memory checked there), ties repeated.  Device pointers;
 * d_sorted_out holds T*K*nS doubles (2.05 GB at nS = 5 000, T = 256, K = 200).  SD_ERR_NONFINITE when F holds NaN or
 * +-inf or a projection overflows; SD_ERR_UNSUPPORTED for nS >= 2^31.
 */
int sd_projection_sort_rows_f64_dev(sd_ctx *ctx, const double *dF, int64_t nS, int64_t T, int d, const double *U,
                                    int64_t K, double *d_sorted_out);

/* New curves dF_new [nY, T, d] against that index, the same U [K, d].  With b / a the reference projections of row
 * (t, k) strictly below / above the new projection y:
 *   tukey:        d_count_out[g] = sum_t min_k (nS + 1 - max(b, a))  == sd_projection_tukey_f64 of S + [g], entry nS
 *   outlyingness: d_o_out[t*nY + g] = max_k |y - med'| / MAD', med' / MAD' of the row with y appended
 *                 == sd_projection_outlyingness_f64 of S + [g], column nS, bit for bit.
 * Device pointers.  SD_ERR_NONFINITE when F_new holds NaN or +-inf or a projection of it overflows;
 * SD_ERR_UNSUPPORTED for nS + 1 >= 2^31. */
int sd_projection_tukey_sorted_f64_dev(sd_ctx *ctx, const double *d_sorted, int64_t nS, int64_t T,
                                       const double *dF_new, int64_t nY, int d, const double *U, int64_t K,
                                       int64_t *d_count_out);
int sd_projection_outlyingness_sorted_f64_dev(sd_ctx *ctx, const double *d_sorted, int64_t nS, int64_t T,
                                              const double *dF_new, int64_t nY, int d, const double *U, int64_t K,
                                              double *d_o_out);

/* Univariate curves dY [T, nY] (dY[t*ldY + g]) against sorted rows from sd_band_sort_rows_f64_dev (the single
 * direction u = 1): d_count_out[g] == sd_band_halfspace_f64 of [S | g], entry nS; d_o_out [T, nY] ==
 * sd_band_outlyingness_f64 of [S | g], column nS.  Errors as above. */
int sd_band_halfspace_sorted_f64_dev(sd_ctx *ctx, const double *d_sorted, int64_t T, int64_t nS, const double *dY,
                                     int64_t nY, int64_t ldY, int64_t *d_count_out);
int sd_band_outlyingness_sorted_f64_dev(sd_ctx *ctx, const double *d_sorted, int64_t T, int64_t nS,
                                        const double *dY, int64_t nY, int64_t ldY, double *d_o_out);

/*
 * Functional spatial depth (L2 spatial depth of curves, Chakraborty & Chaudhuri 2014).  A curve is the vector of its
 * F = T*d values in (t, c) order; r_out[q] = || sum_{j : x_j != x_q} (x_j - x_q) / ||x_j - x_q|| || (Euclidean norms
 * over all F values; duplicates of x_q, and pairs whose squared distance underflows to 0, contribute 0).  The depth is
 * 1 - r / n_pop with n_pop = n in sample and nS + 1 out of sample; the host forms it.
 * layout SD_LAYOUT_NT: X[i*F + f], curve i a row (frames [N, T, d]); SD_LAYOUT_TN: X[f*n + i], curve i a column (the
 * values of a univariate T x n DataFrame), transposed on the device.  Each query's sums run in an order fixed by the
 * indices and the tile sizes alone, so results never depend on the other queries; out of sample r_out[g] equals the
 * in-sample r of S + [g] at entry nS bit for bit.
 * SD_ERR_NONFINITE when an input holds NaN or +-inf, SD_ERR_OVERFLOW when a squared distance overflows (||x_j - x_q||
 * of about 1.3e154 or more).
 */
int sd_spatial_norms_f64(sd_ctx *ctx, const double *X, int64_t n, int64_t F, int layout, const int64_t *query_idx,
                         int64_t nq, double *r_out);
/* new curves Y [nY] against the sample S [nS] (same layout, each dense: S[i*F + f] or S[f*nS + i]) */
int sd_spatial_norms_of_f64(sd_ctx *ctx, const double *S, int64_t nS, const double *Y, int64_t nY, int64_t F,
                            int layout, double *r_out);
/* same with DEVICE pointers, curves as rows only (dS [nS, F], dY [nY, F]); d_r_out holds nY doubles */
int sd_spatial_norms_of_f64_dev(sd_ctx *ctx, const double *dS, int64_t nS, const double *dY, int64_t nY, int64_t F,
                                double *d_r_out);

/*
 * Batched band depth over sub-populations of one matrix (K-sampled blocks, homogeneity
 * permutations): membership[b*n + c] != 0 selects the curves of batch b; queries[b*nqb + i] is
 * the i-th query curve of batch b (must be a member).  count_out[b*nqb + i] as in
 * sd_band_depth_f64 with n replaced by the batch's member count.  One launch sequence for all
 * batches.  X host, layout SD_LAYOUT_TN.
 */
int sd_band_depth_batched_f64(sd_ctx *ctx, const double *X, int64_t T, int64_t n, int64_t ld,
                              const uint8_t *membership, int64_t B, const int64_t *queries,
                              int64_t nqb, int j, int relax, int64_t *count_out);

#ifdef __cplusplus
}
#endif
#endif /* STATDEPTH_B200_H */
