// common.cuh -- shared host/device plumbing of libsdepth.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <functional>

#include "../../include/statdepth_b200.h"

namespace sd {

typedef long long i64;
typedef unsigned long long u64;
typedef unsigned int u32;

void set_error(const char *fmt, ...);

#define SD_CUDA(call)                                                                            \
    do {                                                                                         \
        cudaError_t _e = (call);                                                                 \
        if (_e != cudaSuccess) {                                                                 \
            sd::set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(_e)); \
            return SD_ERR_CUDA;                                                                  \
        }                                                                                        \
    } while (0)

#define SD_TRY(call)                \
    do {                            \
        int _s = (call);            \
        if (_s != SD_OK) return _s; \
    } while (0)

#define SD_REQUIRE(cond, ...)         \
    do {                              \
        if (!(cond)) {                \
            sd::set_error(__VA_ARGS__); \
            return SD_ERR_INVALID;    \
        }                             \
    } while (0)

// Grow-only device buffer owned by the context.
struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    int reserve(size_t bytes);
    void release();
    template <typename T>
    T *as() const { return reinterpret_cast<T *>(p); }
};

// workspace slots of a context
enum BufId {
    BUF_IN = 0,     // device copy of the caller's host input
    BUF_IN2,        // transposed / secondary input
    BUF_QIDX,       // query indices
    BUF_OUT,        // result staging
    BUF_ACC,        // int64 accumulators (MBD: acc_j2[n], acc_j3[n])
    BUF_SPLIT,      // MBD: per-row splitters
    BUF_CURSOR,     // MBD: per-(row, part) fill counts + per-row overflow flags
    BUF_PART_X,     // MBD: partitioned values  / fallback sort scratch
    BUF_PART_J,     // MBD: partitioned curve ids
    BUF_MASK,       // strict BD: per-query sign masks
    BUF_MISC,       // small odds and ends
    BUF_AUX,        // batched / extra
    BUF_WORK,       // MBD: work list of big parts
    BUF_RANKS,      // strict BD matcher: per-time-point ranks of all curves (packed pairs)
    BUF_GEOM,       // Oja counting: the pool's points and the queries' positions inside the pool
    BUF_SLAB,       // MBD slab path: per-row maps, bucket tables, bin starts
    BUF_KEYS,       // extremal depth: per-curve sorted extremities, u32 [n][T] (none of the above is used with it)
    BUF_ORDER,      // extremal depth: curve ids, group starts, merge-sort / scan temp storage
    BUF_PROJ,       // projection depths: projected rows Y
    BUF_PSORT,      // projection depth: sorted rows of Y
    BUF_PRED,       // projection depths: running min / max across direction blocks, per-row med / MAD
    BUF_SPATIAL,    // spatial depth: one row block of weights W [rows][nS] and the per-feature-block partial norms
    NUM_BUFS
};

// status bits written by kernels into ctx->d_status
enum { ST_NONFINITE = 1, ST_INTERNAL = 2, ST_NO_MEMBER = 4, ST_BAD_INPUT = 8, ST_OVERFLOW = 16 };  // ST_BAD_INPUT: caller data out of range

__host__ __device__ static inline i64 ceil_div(i64 a, i64 b) { return (a + b - 1) / b; }

// C(m, J) for J = 2, 3 in int64 (the band-depth j-terms of the out-of-sample kernels)
__device__ __forceinline__ i64 oos_comb(const i64 m, const int J) {
    if (J == 2) return m * (m - 1) / 2;
    return m < 3 ? 0 : (m * (m - 1) / 2) * (m - 2) / 3;  // as comb3_dev (mbd.cu): the product is divisible by 3
}

// order-preserving map double -> u64 (with -0.0 folded onto +0.0 so that == ties stay ties)
__host__ __device__ static inline u64 sortable_key(double x) {
    if (x == 0.0) x = 0.0;
#ifdef __CUDA_ARCH__
    u64 b = (u64)__double_as_longlong(x);
#else
    u64 b;
    memcpy(&b, &x, 8);
#endif
    const u64 mask = (u64)(-(i64)(b >> 63)) | 0x8000000000000000ull;
    return b ^ mask;
}

}  // namespace sd

struct sd_ctx {
    int device = 0;
    int sm_count = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t copy_stream = nullptr;                         // H2D of row blocks overlapped with ranking
    cudaEvent_t ev_pipe[4] = {nullptr, nullptr, nullptr, nullptr};  // copied[2], consumed[2]
    void *stage[2] = {nullptr, nullptr};                        // pinned staging of pageable host input (api.cu)
    size_t stage_cap[2] = {0, 0};
    cudaEvent_t ev_stage[2] = {nullptr, nullptr};
    cudaEvent_t ev_slab[2] = {nullptr, nullptr};                // MBD slab path: table / hist kernel done (mbd.cu)
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};  // h2d start | kernels start | kernels end | d2h end
    sd_timings last = {0, 0, 0, 0, 0, 0};
    int bd_impl = SD_BD_AUTO;
    int mbd_force_fallback = 0;
    int mbd_no_wait = 0;    // set around pipelined host calls: mbd_all_device must not wait for device results
    int profile = 0;
    int simplicial_impl = SD_SIMPLICIAL_AUTO;
    int async_device = 0;   // SD_OPT_ASYNC_DEVICE
    int pending = 0;        // an asynchronous device call has been queued and not yet completed by sd_sync()
    static const int MAX_PROF = 256;                 // event pairs per call when profiling
    cudaEvent_t prof_ev[2 * MAX_PROF] = {};          // created lazily
    int prof_phase[MAX_PROF] = {};
    int prof_n = 0;
    int64_t phase_ns[SD_PHASE_COUNT] = {};
    sd::DevBuf buf[sd::NUM_BUFS];
    int *d_status = nullptr;  // device int[8]: [0] status bits, [1] MBD rows ranked by the generic path; [6..7] mbd.cu
    int *h_status = nullptr;  // pinned mirror; [2] and [3] also receive the slab path's unfit-row counts mid-call (mbd.cu)
    int *h_status_dev = nullptr;  // the mirror as kernels address it (mapped), for the counts the slab kernels store
    int mbd_attributes_set = 0;   // the rank pipeline's kernel attributes are set on this context's device (mbd.cu)
};

namespace sd {

// timing helpers: record the four phase boundaries of a host-buffer call
int begin_call(sd_ctx *ctx);                 // resets status, records ev[0]
int mark(sd_ctx *ctx, int which);            // records ev[which]
int end_call(sd_ctx *ctx, bool had_copies);  // syncs, fills ctx->last, maps status bits to errors
int check_status(sd_ctx *ctx);               // (after sync) translate *h_status
// profiling brackets (no-ops unless SD_OPT_PROFILE): prof_begin before a phase's launches, prof_end after
int prof_begin(sd_ctx *ctx, int phase);
int prof_end(sd_ctx *ctx);

// kernels / drivers implemented in the other translation units (all stream-ordered on ctx->stream)
int band_depth_device(sd_ctx *ctx, const double *dX, i64 T, i64 n, i64 ld, const i64 *d_q, i64 nq, int j,
                      int relax, i64 *d_out);
// The int64 guard of relaxed band depth with `others` curves besides the one ranked (n - 1 within a sample, nS out
// of sample): T * C(others, j) must fit, and for j = 3 also 3 * C(others, 3).  relaxed_overflow_check sets the error
// (prefixed by who) and returns SD_ERR_OVERFLOW (api.cu).
bool relaxed_overflows(i64 T, i64 others, int j);
int relaxed_overflow_check(i64 T, i64 others, int j, const char *who);
// K1, the per-row strict ranks of X [T, n] (mbd.cu).  mbd_all_device: d_acc2[c] (and d_acc3[c], if given) = the
// relaxed j = 2 (3) numerator summed over the rows, added to the old value if `accumulate` (row blocks of one
// matrix); group_rows = g > 0: T / g matrices of g rows accumulate into the rows of [T / g][n] (batched permutations).
int mbd_all_device(sd_ctx *ctx, const double *dX, i64 T, i64 n, i64 ld, i64 *d_acc2, i64 *d_acc3,
                   bool accumulate = false, i64 group_rows = 0);
// d_rank_b / d_rank_a[t*n + c] = #other values of row t strictly below / above X[t, c]; d_rank_a may be null.
int rank_rows_device(sd_ctx *ctx, const double *dX, i64 T, i64 n, i64 ld, int *d_rank_b, int *d_rank_a);
// int32 workspace for rank-only passes in row blocks of *RB rows (ints_per_row each) within a fixed budget
int rank_block_workspace(sd_ctx *ctx, i64 T, i64 ints_per_row, i64 *RB, int **ws);
// Rank-only passes in blocks of that workspace, at most max_rows each: consume(r0, rows, rb, ra) queues the caller's
// reduction of one block's ranks (ra null unless want_a) and counts its launches.
using RankBlockFn = std::function<void(i64 r0, i64 rows, const int *rb, const int *ra)>;
int for_each_rank_block(sd_ctx *ctx, const double *dX, i64 T, i64 n, i64 ld, bool want_a, i64 max_rows,
                        const RankBlockFn &consume);
// K2, strict band depth (bd_bits.cu, bd_gemm.cu, bd_match.cu; strict_enumerate in api.cu): d_q must not be null.
// The strict branch of band_depth_device writes the ids 0 .. nq - 1 into BUF_QIDX when the caller gives no query
// list, so no strict driver may reserve BUF_QIDX (growing it would free that list).
int bd_strict_device(sd_ctx *ctx, const double *dX, i64 T, i64 n, i64 ld, const i64 *d_q, i64 nq, int j,
                     i64 *d_out, u64 *d_hits = nullptr);
int bd_strict_gemm_device(sd_ctx *ctx, const double *dX, i64 T, i64 n, i64 ld, const i64 *d_q, i64 nq,
                          i64 *d_out);
int probe_int8_peak(sd_ctx *ctx, double *ops_per_s);
bool bd_match_supported(i64 T, i64 n);
// the enumerating strict J = 2 path (strict_enumerate) that recomputes the queries the matcher cannot certify
using StrictFallback = int (*)(sd_ctx *ctx, const double *dX, i64 T, i64 n, i64 ld, const i64 *d_q, i64 nq,
                               i64 *d_out);
int bd_strict_match_device(sd_ctx *ctx, const double *dX, i64 T, i64 n, i64 ld, const i64 *d_q, i64 nq, i64 *d_out,
                           StrictFallback fallback, i64 *n_fallback);
int bd_strict_match_batched_device(sd_ctx *ctx, const double *dXg, i64 nb, i64 T, i64 n, const i64 *d_ql, i64 nqb,
                                   i64 *d_out, StrictFallback fallback);
int transpose_device(sd_ctx *ctx, const double *d_in, i64 rows, i64 cols, i64 ld_in, double *d_out);
int gather_i64_device(sd_ctx *ctx, const i64 *d_src, const i64 *d_idx, i64 nq, i64 *d_out);
int compact_columns_device(sd_ctx *ctx, const double *dX, i64 T, i64 n, const i64 *d_cols, i64 m, double *d_out);
int compact_batches_device(sd_ctx *ctx, const double *dX, i64 T, i64 n, const i64 *d_cols, i64 m, i64 nb,
                           double *d_out);
int l1_device(sd_ctx *ctx, const double *dP, i64 n, int d, const i64 *d_q, i64 nq, double *d_out,
              i64 n_pop = 0);
int oja_device(sd_ctx *ctx, const double *dP, i64 n, int d, const i64 *d_q, i64 nq, const i64 *d_pool,
               i64 npool, double hull_volume, double *d_out);
int cloud_blocks_device(sd_ctx *ctx, const double *dP, int d, const i64 *d_member, const i64 *d_off,
                        const i64 *d_qpos, i64 B, int kind, double tol, const double *d_volume, double *d_out);
int simplicial_device(sd_ctx *ctx, const double *dP, i64 n, int d, const i64 *d_q, i64 nq, double tol,
                      i64 *d_out, bool oos = false);
// what simplicial2_count_device reduces the two rank passes of the angular keys to (simplicial_count.cu)
enum ScReduce { SC_TRIANGLES, SC_HALFSPACE };
int simplicial2_count_device(sd_ctx *ctx, const double *d_pts, i64 n, i64 stride_j, i64 T, const i64 *d_q, i64 nq,
                             double tol, i64 *d_out, i64 m_others = -1, ScReduce reduce = SC_TRIANGLES);
// halfspace depth, d = 1 (halfspace.cu): d_out[c] = sum_t (n - max(b_t(c), a_t(c))) over the rows of X [T, n]
int halfspace1_device(sd_ctx *ctx, const double *dX, i64 T, i64 n, i64 ld, i64 *d_out);
// random projection depths (projection.cu): dU == nullptr takes the rows of X [T, N] (leading dimension ldX) as
// the projections of the single direction u = 1.  PJ_TUKEY: d_count [N] = sum_t min_k (N - max(b, a)).
// PJ_OUTLYING: d_o [T][N] = max_k |y - med| / MAD; med_out / mad_out [T][K] (copied with out_kind) may be NULL.
enum ProjKind { PJ_TUKEY, PJ_OUTLYING };
int projection_device(sd_ctx *ctx, const double *dF, i64 N, i64 T, int d, i64 ldX, const double *dU, i64 K,
                      ProjKind kind, i64 *d_count, double *d_o, double *med_out, double *mad_out,
                      cudaMemcpyKind out_kind);
// projection.cu's row blocks, shared by the fitted projected references (reference_proj.cu): rows of N projections
// (leading dimension N rounded up to even) that fit PJ_BUDGET; kb_max directions by tb_max time points per block (a
// time block keeps all K directions when K rows fit); project_device writes the block (t0 .. t0 + tb, kb directions
// from dU) as Y[(tt * kb + kk) * ldY + i].
i64 projection_rows_max(i64 N);
void projection_blocks(i64 rows_max, i64 T, i64 K, i64 *kb_max, i64 *tb_max);
int project_device(sd_ctx *ctx, const double *dF, i64 N, i64 T, int d, const double *dU, i64 kb, i64 t0, i64 tb,
                   double *Y, i64 ldY);
// fitted projected references (reference_proj.cu, K13): d_sorted[(t * K + k) * nS + j] = the j-th smallest of the
// projections y_k(., t) of the nS reference curves F [nS, T, d]
int projection_sort_rows_device(sd_ctx *ctx, const double *dF, i64 nS, i64 T, int d, const double *dU, i64 K,
                                double *d_sorted);
// new observations against such an index: dU == nullptr takes the rows of Y [T, nY] (leading dimension ldY) against
// K9's sorted rows (K = 1, y = x); else dY holds new curves [nY, T, d].  PJ_TUKEY: d_count [nY] = sum_t min_k
// (nS + 1 - max(b, a)); PJ_OUTLYING: d_o [T][nY] = max_k |y - med'| / MAD' of the row with y appended.
int projection_sorted_device(sd_ctx *ctx, const double *d_sorted, i64 nS, i64 T, const double *dY, i64 nY, i64 ldY,
                             int d, const double *dU, i64 K, ProjKind kind, i64 *d_count, double *d_o);
// functional spatial depth (spatial.cu, K14): d_r[q] = || sum_s u(S_s - Q_q) || of the rows Q[idx(q) * F] (idx = d_qidx
// or q) against the sample rows dS [nS, F], in an order fixed by q's index and the tile sizes; ST_OVERFLOW when a
// squared distance overflows
int spatial_device(sd_ctx *ctx, const double *dQ, const i64 *d_qidx, i64 nq, const double *dS, i64 nS, i64 F,
                   double *d_r);
// out-of-sample depth (oos.cu): pooled inputs, sample first, queries after it
int band_depth_oos_device(sd_ctx *ctx, const double *dX, i64 T, i64 nS, i64 nY, i64 ld, int j, int relax,
                          i64 *d_out);
// sorted reference rows and out-of-sample counts from them (reference.cu)
int sort_rows_device(sd_ctx *ctx, const double *dX, i64 T, i64 nS, i64 ld, double *d_sorted);
int depth_sorted_device(sd_ctx *ctx, const double *d_sorted, i64 T, i64 nS, const double *dY, i64 nY, i64 ldY,
                        int J, i64 *d_out);
// outlier detection (outliers.cu)
int rank_sums_device(sd_ctx *ctx, const double *dX, i64 T, i64 n, i64 ld, i64 *d_q, i64 *d_b, i64 *d_a);
int envelope_device(sd_ctx *ctx, const double *dX, i64 T, i64 n, i64 ld, const uint8_t *d_member, double factor,
                    double *d_lower, double *d_upper, i64 *d_outside);
// extremal depth (extremal.cu): m = |b - a| of rows, and the numerators e from the full m
int extremity_device(sd_ctx *ctx, const double *dX, i64 T, i64 n, i64 ld, int *d_m);
int extremal_depth_device(sd_ctx *ctx, const int *d_m, i64 T, i64 n, i64 *d_e);
int iota_from_device(sd_ctx *ctx, i64 *d_p, i64 count, i64 base);
int finite_check_device(sd_ctx *ctx, const double *dX, i64 rows, i64 cols, i64 ld);
int oja2_count_device(sd_ctx *ctx, const double *d_pts, i64 n, const i64 *d_q, i64 nq, double hull_volume,
                      double *d_out);
int simplex_depth_device(sd_ctx *ctx, const double *dF, i64 N, i64 T, int d, const i64 *d_q, i64 nq,
                         int relax, double tol, i64 *d_out);

}  // namespace sd
