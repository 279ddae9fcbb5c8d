// sorted_row.cuh -- searches in one sorted row, shared by the fitted-reference kernels (reference.cu, K9, and
// reference_proj.cu, K13) and projection depth's median / MAD (projection.cu, K12).
//
// A row is read through an accessor, so that one selection serves a plain sorted row and the virtual row of an
// out-of-sample query (the reference's sorted row with the new value inserted, never materialised).
#pragma once
#include <math.h>

#include "common.cuh"

namespace sd {

// b = #values of the sorted row[0..n) strictly below y, a = #values strictly above: a lower-bound (first >= y) and an
// upper-bound (first > y) search in the same loop.  Their step sizes depend on n only, so the two chains of dependent
// loads interleave and no warp diverges.  Every read stays in [0, n) and b, a in [0, n] whatever the row holds.
__device__ __forceinline__ void sorted_bounds(const double *row, const i64 n, const double y, i64 &b, i64 &a) {
    const double *lo = row, *hi = row;
    for (i64 len = n; len > 1;) {
        const i64 half = len >> 1;
        lo = lo[half] < y ? lo + half : lo;
        hi = hi[half] <= y ? hi + half : hi;
        len -= half;
    }
    b = (lo - row) + (*lo < y);
    a = n - ((hi - row) + (*hi <= y));
}

// a sorted row in memory
struct PlainRow {
    const double *s;
    __device__ __forceinline__ double operator[](const i64 k) const { return s[k]; }
};

// the sorted row s[0..n) with y inserted at p = #{s < y}: v[k] = s[k] (k < p), y (k = p), s[k - 1] (k > p).  For
// 0 <= p <= n and k in [0, n], every read of s stays in [0, n).
struct InsertedRow {
    const double *__restrict__ s;
    i64 p;
    double y;
    __device__ __forceinline__ double operator[](const i64 k) const { return k < p ? s[k] : (k == p ? y : s[k - 1]); }
};

// k-th smallest (0-based) of L ∪ R, L[j] = |s[m-1-j] - med| (j < m), R[j] = |s[m+j] - med| (j < n - m): i = how
// many of the k + 1 smallest come from L, the least i with R[k - i] <= L[i].  Both lists are non-decreasing because
// rounding is monotone, so a binary search over i finds it in O(log n).
template <class Row>
__device__ __forceinline__ double kth_deviation(const Row &s, const i64 n, const i64 m, const double med, const i64 k) {
    const i64 nL = m, nR = n - m;
    i64 lo = k + 1 - nR > 0 ? k + 1 - nR : 0;
    i64 hi = k + 1 < nL ? k + 1 : nL;
    while (lo < hi) {
        const i64 i = (lo + hi) >> 1, j = k + 1 - i;
        if (j > 0 && i < nL && fabs(__dsub_rn(s[m + j - 1], med)) > fabs(__dsub_rn(s[m - 1 - i], med))) lo = i + 1;
        else hi = i;
    }
    const i64 j = k + 1 - lo;
    double v = 0.0;
    if (lo > 0) v = fabs(__dsub_rn(s[m - lo], med));
    if (j > 0) {
        const double r = fabs(__dsub_rn(s[m + j - 1], med));
        if (lo == 0 || r > v) v = r;
    }
    return v;
}

// med and MAD of the sorted row s[0..n) exactly as np.median and np.median(np.abs(s - med)) (unscaled MAD)
template <class Row>
__device__ __forceinline__ double row_median(const Row &s, const i64 n) {
    const i64 h = n >> 1;
    return (n & 1) ? s[h] : __ddiv_rn(__dadd_rn(s[h - 1], s[h]), 2.0);
}

template <class Row>
__device__ __forceinline__ double row_mad(const Row &s, const i64 n, const double md) {
    const i64 h = n >> 1;
    i64 m = 0;  // #values < md: lower bound
    for (i64 len = n; len > 0;) {
        const i64 half = len >> 1;
        if (s[m + half] < md) {
            m += half + 1;
            len -= half + 1;
        } else {
            len = half;
        }
    }
    return (n & 1) ? kth_deviation(s, n, m, md, h)
                   : __ddiv_rn(__dadd_rn(kth_deviation(s, n, m, md, h - 1), kth_deviation(s, n, m, md, h)), 2.0);
}

// |y - med| / MAD; MAD = 0 gives 0 where y == med and +inf elsewhere
__device__ __forceinline__ double outlyingness(const double y, const double md, const double s) {
    return s == 0.0 ? (y == md ? 0.0 : (double)INFINITY) : __ddiv_rn(fabs(__dsub_rn(y, md)), s);
}

}  // namespace sd
