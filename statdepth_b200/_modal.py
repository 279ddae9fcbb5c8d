"""h-modal depth on the B200 engine (csrc/modal.cu, DESIGN.md K15): the kernel depth of curves of Cuevas, Febrero &
Fraiman (2007) (depth.mode in fda.usc), with the Gaussian kernel.

A curve is the vector of its F = T d values in (t, c) order, compared by the plain Euclidean norm over all F values, as
in K14 (a uniform time weight would cancel between the distances and a quantile bandwidth).  With phi the standard
normal density:

    MD(x_q) = (1 / n) sum_j phi(||x_j - x_q|| / h)

j runs over all n curves, x_q included, so the depth lies in [phi(0) / n, phi(0)].  The engine returns
S_q = sum_j exp(c d2_qj) with c = -0.5 / (h * h); the host forms S_q / n * phi(0).  The bandwidth is given, or it is
np.quantile of the n (n - 1) / 2 pair distances (method 'linear'): the engine selects the two order statistics of the
squared distances the quantile needs (sqrt is monotone and correctly rounded, so their roots are those of the
distances), and the host applies numpy's index and interpolation arithmetic to them, so h equals np.quantile bit for
bit whenever the squared distances are equal.  Out of sample a new curve g is scored against the sample S with S's
bandwidth and the divisor n_S + 1: FunctionalModalDepth(S + [g], bandwidth=h) gives g the same bits.

Sharding under `enable_distributed()`: every rank selects the bandwidth from the whole sample (the same bits as one
process) and scores its block of the queries (`_dist.query_sharded`).
"""
import math
from typing import List

import numpy as np
import pandas as pd

from . import _dist
from ._engine import get_engine, resident
from ._functional import _positions
from ._spatial import _checked_new_curves, _rows, _spatial_curves

__all__ = ['DEFAULT_QUANTILE', '_checked_bandwidth', '_quantile_bandwidth', '_functional_modal',
           '_functional_modal_of', '_ModalReference']

DEFAULT_QUANTILE = 0.15
PHI0 = 1.0 / math.sqrt(2.0 * math.pi)  # phi(0)


def _checked_bandwidth(quantile, bandwidth):
    """The bandwidth as given (a float), or None when it is to be selected at `quantile`; ValueError for a quantile
    outside [0, 1], for both given, and for a bandwidth that is not finite and > 0 or whose square is not a finite
    normal number."""
    if bandwidth is not None:
        if quantile != DEFAULT_QUANTILE:
            raise ValueError('pass quantile or bandwidth, not both (a given bandwidth ignores the quantile)')
        h = float(bandwidth)
        if not (math.isfinite(h) and h > 0.0 and math.isfinite(h * h) and h * h >= np.finfo(np.float64).tiny):
            raise ValueError('bandwidth must be finite and > 0, with a finite normal square (got %r)' % (bandwidth,))
        return h
    q = float(quantile)
    if not 0.0 <= q <= 1.0:
        raise ValueError('quantile must lie in [0, 1] (got %r)' % (quantile,))
    return None


def _quantile_bandwidth(N: int, quantile: float, order_stats) -> float:
    """np.quantile(D, quantile) of N sorted values D without D: order_stats(k) gives (D[k], D[min(k + 1, N - 1)]).
    numpy's own arithmetic for method 'linear' (its virtual index (N - 1) q, the floor and gamma of _get_indexes and
    _get_gamma, and _lerp with its t >= 0.5 branch), in the same float64 operations."""
    q = float(quantile)
    v = (N - 1) * q
    if v >= N - 1:  # numpy takes the last value on both sides (index -1)
        k, prev = N - 1, -1
    else:
        k = prev = int(math.floor(v))
    a, b = order_stats(k)
    if prev == -1:
        b = a
    t = v - prev
    diff = b - a
    h = a + diff * t
    if t >= 0.5:
        h = b - diff * (1 - t)
    return float(h)


def _selected_bandwidth(eng, A, n: int, quantile: float) -> float:
    """The bandwidth at `quantile` of the pair distances of the n curves A (rows, as eng reads them)."""
    if n < 2:
        raise ValueError('one curve has no pair distances to take a bandwidth from: pass bandwidth=')

    def order_stats(k):
        d2 = eng.modal_pair_select(A, k)
        return float(np.sqrt(d2[0])), float(np.sqrt(d2[1]))

    h = _quantile_bandwidth(n * (n - 1) // 2, quantile, order_stats)
    if not (h * h >= np.finfo(np.float64).tiny):
        raise ValueError('the bandwidth at quantile %r of the pair distances is %r (at least that share of the pairs '
                         'are duplicates, or nearly): pass bandwidth=' % (quantile, h))
    return h


def _functional_modal(data: List[pd.DataFrame], to_compute=None, quantile=DEFAULT_QUANTILE,
                      bandwidth=None) -> pd.Series:
    """[df] (T x n, curves are columns; to_compute = column labels) or N DataFrames of T x d (one curve each;
    to_compute = list positions)."""
    h = _checked_bandwidth(quantile, bandwidth)
    X, F = _spatial_curves(data)
    A = _rows(X, F)
    n = A.shape[0]
    labels = (data[0].columns if X is not None else pd.RangeIndex(n)) if to_compute is None else to_compute
    axis = data[0].columns if X is not None else pd.RangeIndex(n)
    q = _positions(labels, axis, 'to_compute')
    eng = get_engine()
    R = resident(eng, A)  # one upload for both passes
    if h is None:
        h = _selected_bandwidth(eng, R, n, quantile)
    c = -0.5 / (h * h)
    s = _dist.query_sharded(lambda qb: eng.modal_sums(R, c, qb), q, np.float64)
    index = list(labels) if X is None else labels
    return pd.Series(index=index, data=np.asarray(s, dtype=np.float64) / n * PHI0)


def _functional_modal_of(data: List[pd.DataFrame], sample: List[pd.DataFrame], quantile=DEFAULT_QUANTILE,
                         bandwidth=None) -> pd.Series:
    """Depth of the new curves data against sample, each as if appended alone to it, with sample's bandwidth."""
    h = _checked_bandwidth(quantile, bandwidth)
    XS, FS = _spatial_curves(sample)
    X, F = _checked_new_curves(data, XS, FS)
    ref = _ModalReference(X=XS, F=FS, quantile=quantile, bandwidth=h)
    try:
        depth = ref.depths(X if X is not None else F)
    finally:
        ref.close()
    index = data[0].columns if X is not None else list(range(len(data)))
    return pd.Series(index=index, data=depth)


class _ModalReference:
    """A sample of curves kept for h-modal depth: n_S x F doubles uploaded once to the engine's device, for as long as
    the reference lives, and its bandwidth, selected once at construction unless given.  Every rank holds all of it."""

    def __init__(self, X=None, F=None, quantile=DEFAULT_QUANTILE, bandwidth=None):
        h = _checked_bandwidth(quantile, bandwidth)
        A = _rows(X, F)
        self.nS, self.F = A.shape
        self.eng = get_engine()
        self.sample = resident(self.eng, A)
        self.bandwidth = h if h is not None else _selected_bandwidth(self.eng, self.sample, self.nS, quantile)
        self.c = -0.5 / (self.bandwidth * self.bandwidth)

    def depths(self, Y: np.ndarray) -> np.ndarray:
        """Depth of every new curve: the columns of Y [T, nY] (univariate), else Y [nY, T, d]; each equals
        FunctionalModalDepth of the sample with that curve appended and bandwidth=self.bandwidth, bit for bit."""
        A = Y.T if Y.ndim == 2 else Y.reshape(Y.shape[0], -1)
        if A.shape[1] != self.F:
            raise ValueError('data and sample must have the same number of values per curve.')
        if A.shape[0] == 0:
            return np.zeros(0, dtype=np.float64)
        s = _dist.query_sharded(lambda qb: self.eng.modal_sums_of(self.sample, A[qb], self.c), np.arange(A.shape[0]),
                                np.float64)
        return np.asarray(s, dtype=np.float64) / (self.nS + 1) * PHI0

    def close(self) -> None:
        self.sample = None
