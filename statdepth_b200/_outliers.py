"""Functional outlier detection drivers: functional boxplot (Sun & Genton 2011), outliergram (Arribas-Gil & Romo
2014) and extremal depth (Narisetty & Nair 2016), built on the integers K1 ranks with (csrc/outliers.cu, DESIGN.md
K8; csrc/extremal.cu, K10).

Both take univariate data X [T, n] (time rows x curves) and return plain arrays; depth.py wraps them in result
objects.  Every per-curve quantity is exact int64 from the engine; floats are formed here once, at the end.

On one GPU the matrix crosses PCIe once per call: the rows are uploaded once (Engine.upload) and every engine call
reads them in place.  Under `enable_distributed()` every rank takes a block of time rows: the rank sums and outside
counts are all-reduced, the per-row envelopes all-gathered, and the whisker pass runs after the outside counts are
reduced.  Extremal depth is not additive over rows: every rank computes the extremities of its rows, they are
all-gathered, and every rank orders the curves on the full matrix.
"""
import math
import numbers
from fractions import Fraction
from typing import List

import numpy as np
import pandas as pd
from scipy.special import binom

from . import _dist
from ._engine import get_engine, resident
from ._functional import _values
from ._helper import _handle_depth_errors

__all__ = ['_checked_values', '_check_central', '_check_extremal_rows', '_functional_boxplot', '_outliergram',
           '_extremal_depth']

EXTREMAL_T_MAX = 16384  # SD_EXTREMAL_T_MAX (include/statdepth_b200.h): the bound of the per-curve sort on the GPU


def _real(x) -> bool:
    return isinstance(x, numbers.Real) and not isinstance(x, bool)


NO_FACTOR = object()  # _checked_values without the outlier factor (None is a bad factor, not a missing one)


def _checked_values(data: List[pd.DataFrame], factor, deep_check=False,
                    what='functional outlier detection') -> np.ndarray:
    """The validation of FunctionalDepth([df], J=2, relax=True), then the outlier factor (unless NO_FACTOR);
    X [T, n]."""
    if isinstance(data, list) and len(data) > 1:
        raise NotImplementedError('%s is implemented for univariate data ([DataFrame])' % what)
    _handle_depth_errors(data=data, J=2, containment='r2', relax=True, deep_check=deep_check)
    if factor is not NO_FACTOR and not (_real(factor) and math.isfinite(factor) and factor >= 0):
        raise ValueError('factor must be a finite number >= 0.')
    X = _values(data[0])
    if X.shape[1] < 2:
        raise ValueError('%s needs at least two curves.' % what)
    return X


def _check_extremal_rows(T: int) -> None:
    if T > EXTREMAL_T_MAX:
        raise NotImplementedError('extremal depth is implemented for up to %d time points (got %d)'
                                  % (EXTREMAL_T_MAX, T))


def _check_central(central) -> None:
    if not (_real(central) and 0 < central <= 1):
        raise ValueError('central must be a number in (0, 1].')


class _Rows:
    """A block of time rows X [T, n], resident on its engine (an empty block is never uploaded)."""

    def __init__(self, eng, X):
        self.eng = eng
        self.T, self.n = X.shape
        self.X = resident(eng, X) if self.T > 0 else X

    def mbd_counts(self) -> np.ndarray:
        """Q [n]: the relaxed J = 2 numerators of these rows."""
        if self.T == 0:
            return np.zeros(self.n, dtype=np.int64)
        return self.eng.band_depth_counts(self.X, None, 2, True)

    def rank_sums(self):
        """(Q, B) [n]: numerators and sums of the curves strictly below, over these rows."""
        if self.T == 0:
            return np.zeros(self.n, dtype=np.int64), np.zeros(self.n, dtype=np.int64)
        return self.eng.band_rank_sums(self.X)

    def extremity(self) -> np.ndarray:
        """m [T, n] int32: the pointwise extremities |b - a| of these rows, where the rows are (on one GPU they never
        reach the host)."""
        if self.T == 0:
            return np.zeros((0, self.n), dtype=np.int32)
        return self.eng.band_extremity(self.X)

    def envelope(self, member: np.ndarray, factor: float, want_outside: bool):
        """(lo [T], hi [T], outside [n] or None) of these rows over the member curves."""
        if self.T == 0:
            return np.zeros(0), np.zeros(0), (np.zeros(self.n, dtype=np.int64) if want_outside else None)
        return self.eng.band_envelope(self.X, member, factor, want_outside)


def _local_rows(X: np.ndarray):
    """(this rank's rows of X on its engine, world size)."""
    rank, size = _dist.world()
    lo, hi = _dist.block(X.shape[0], rank, size)
    return _Rows(get_engine(), X[lo:hi]), size


def _summed(a: np.ndarray, size: int) -> np.ndarray:
    return a if size == 1 else _dist.allreduce(np.asarray(a, dtype=np.int64))


def _gathered(a: np.ndarray, T: int, size: int) -> np.ndarray:
    return a if size == 1 else _dist.allgather_blocks(np.asarray(a, dtype=np.float64), T)


def _mbd(q: np.ndarray, T: int, n: int) -> np.ndarray:
    """The arithmetic of _functional._univariate_depths for relax=True, J=2: bit-identical to FunctionalDepth."""
    depth = np.zeros(n, dtype=np.float64)
    s = q.astype(np.float64) / float(T)
    return depth + s / binom(n, 2)


def fences(lo: np.ndarray, hi: np.ndarray, factor: float):
    """(lower, upper) = (lo - f, hi + f), f = factor * (hi - lo): the rounded operations the kernel counts with."""
    f = np.multiply(factor, np.subtract(hi, lo))
    return np.subtract(lo, f), np.add(hi, f)


def central_count(central: float, n: int) -> int:
    """k = ceil(central * n) >= 1, taken on the exact value of the double `central` (0.3 * 10 is 3, not 4)."""
    return max(1, math.ceil(Fraction(central) * n))


def _extremal_numerators(rows: _Rows, T: int, size: int) -> np.ndarray:
    """e [n] of the whole matrix X [T, n] from this rank's rows (a collective when size > 1)."""
    m = rows.extremity()
    return rows.eng.extremal_depth(m if size == 1 else _dist.allgather_blocks(m, T))


def _extremal_depth(X: np.ndarray) -> np.ndarray:
    """Extremal-depth numerators e [n] of the curves of X [T, n]: ED = e / n."""
    rows, size = _local_rows(X)
    return _extremal_numerators(rows, X.shape[0], size)


def _functional_boxplot(X: np.ndarray, factor: float, central: float, depth: str = 'mbd') -> dict:
    """Central region: the ceil(central * n) curves of largest MBD numerator Q (depth='mbd') or extremal-depth
    numerator e (depth='extremal'), ties by column position.  Envelope of the central region per row, fences inflated
    by factor * its width, outside counts against the fences, and the whiskers: the envelope of every curve that
    never leaves the fences."""
    T, n = X.shape
    rows, size = _local_rows(X)
    if depth == 'extremal':
        q = _extremal_numerators(rows, T, size)
        depths = q.astype(np.float64) / n
    else:
        q = _summed(rows.mbd_counts(), size)
        depths = _mbd(q, T, n)
    order = np.argsort(-q, kind='stable')  # Q (or e) descending, then column position ascending
    central_pos = order[:central_count(central, n)]
    member = np.zeros(n, dtype=np.uint8)
    member[central_pos] = 1
    lo, hi, outside = rows.envelope(member, factor, True)
    lo, hi = _gathered(lo, T, size), _gathered(hi, T, size)
    outside = _summed(outside, size)
    inside = (outside == 0).astype(np.uint8)  # never empty for factor >= 0: the central curves are inside
    wlo, whi, _ = rows.envelope(inside, 0.0, False)
    lower, upper = fences(lo, hi, factor)
    return dict(depth=depths, q=q, central=central_pos, envelope=(lo, hi), fences=(lower, upper),
                whiskers=(_gathered(wlo, T, size), _gathered(whi, T, size)), outside=outside)


def outliergram_distance(q: np.ndarray, b: np.ndarray, T: int, n: int):
    """(MEI [n], d [n]) from the exact sums Q and B.

    U = n T - B counts the curves at or above c over all rows, c itself included; MEI = U / (n T).  The paper's
    bound MBD <= a0 + a1 MEI + a2 n^2 MEI^2 (its MBD counts the n - 1 pairs containing c: ours + 2 / n), times
    T^2 C(n, 2), is the integer  D = (n + 1) U T - U^2 - T Q - n T^2 >= 0 on tie-free data.  Its terms reach ~1e16
    at n = 100 000, T = 1024 and cancel, so D is formed in integers (int64 while (n + 1) n T^2 < 2^63 bounds every
    term and partial sum, Python ints beyond) and divided once."""
    if (n + 1) * n * T * T < 2 ** 63:
        U = n * T - b.astype(np.int64)
        D = (n + 1) * U * T - U * U - T * q.astype(np.int64) - n * T * T
    else:
        U = n * T - b.astype(object)
        D = (n + 1) * U * T - U * U - T * q.astype(object) - n * T * T
    mei = U.astype(np.float64) / float(n * T)
    d = D.astype(np.float64) / float(T * T * (n * (n - 1) // 2))
    return mei, d


def _outliergram(X: np.ndarray, factor: float) -> dict:
    """Shape outliers: d >= q3 + factor (q3 - q1), q1 / q3 the 25th / 75th percentiles of d (numpy's linear rule)."""
    T, n = X.shape
    rows, size = _local_rows(X)
    q, b = rows.rank_sums()
    q, b = _summed(q, size), _summed(b, size)
    mei, d = outliergram_distance(q, b, T, n)
    q1, q3 = np.percentile(d, [25, 75])
    return dict(depth=_mbd(q, T, n), q=q, mei=mei, distance=d, outlier=d >= q3 + factor * (q3 - q1))
