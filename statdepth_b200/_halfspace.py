"""Halfspace (Tukey) depth drivers on the B200 engine (csrc/halfspace.cu and hs_reduce_kernel in
csrc/simplicial_count.cu; DESIGN.md K11).

A point p of a sample of n points has the numerator h(p) = the fewest sample points, p included, in a closed
half-plane (d = 2) or half-line (d = 1) whose boundary passes through p, and HD = h / n.  Curves take the
integrated form of Claeskens, Hubert, Slaets & Vakili (2014) with uniform weights: H(c) = sum_t h_t(c), h_t the
numerator of c(t) among the n values at time t, and the depth H / (T n).  The numerators are exact int64 from the
engine; the host divides once.

Sharding under `enable_distributed()`: point clouds and bivariate curves split the queries (`_dist.query_sharded`);
univariate curves split the time rows, whose numerators are additive, and all-reduce them.
"""
from typing import List

import numpy as np
import pandas as pd

from . import _dist
from ._engine import get_engine
from ._functional import _positions, _values

__all__ = ['_pointcloud_halfspace', '_functional_halfspace']


def _pointcloud_halfspace(data: pd.DataFrame, to_compute=None) -> pd.Series:
    """Halfspace depth of the requested rows of the n x d cloud data (d = 1 or 2), indexed by to_compute (all rows,
    data.index, when None)."""
    n, d = data.shape
    if d not in (1, 2):
        raise NotImplementedError('halfspace depth is implemented for d = 1 or 2 on the B200 engine (got d=%d)' % d)
    if to_compute is None:
        to_compute = data.index
    q = _positions(to_compute, data.index, 'to_compute')
    P = np.ascontiguousarray(_values(data))
    eng = get_engine()
    cnt = _dist.query_sharded(lambda qb: eng.halfspace_counts(P, qb), q, np.int64)
    return pd.Series(index=to_compute, data=cnt.astype(np.float64) / n)


def _functional_halfspace(data: List[pd.DataFrame], to_compute=None) -> pd.Series:
    """Integrated halfspace depth: [df] (T x n, curves are columns; to_compute = column labels) or N DataFrames of
    T x 2 (one curve each; to_compute = list positions)."""
    if not isinstance(data, list):
        raise ValueError('data must be passed as a list.')
    if len(data) == 0:
        raise ValueError('No data passed.')
    if len(data) == 1:
        df = data[0]
        T, n = df.shape
        cols = df.columns if to_compute is None else to_compute
        q = None if to_compute is None else _positions(to_compute, df.columns, 'to_compute')
        cnt = _univariate_counts(_values(df))
        if q is not None:
            cnt = cnt[q]
        return pd.Series(index=cols, data=cnt.astype(np.float64) / (T * n))
    channels = {df.shape[1] for df in data}
    if channels != {2}:
        raise NotImplementedError('multivariate halfspace depth is implemented for 2 channels on the B200 engine '
                                  '(got %s)' % sorted(channels))
    if len({df.shape[0] for df in data}) > 1:
        raise ValueError('every curve must have the same number of time points.')
    N, T = len(data), data[0].shape[0]
    f = list(range(N)) if to_compute is None else to_compute
    q = _positions(f, pd.RangeIndex(N), 'to_compute')
    F = np.stack([_values(df) for df in data])
    eng = get_engine()
    cnt = _dist.query_sharded(lambda qb: eng.functional_halfspace_counts(F, qb), q, np.int64)
    return pd.Series(index=f, data=cnt.astype(np.float64) / (T * N))


def _univariate_counts(X: np.ndarray) -> np.ndarray:
    """H [n] of the curves of X [T, n]: this rank's block of time rows, all-reduced across ranks."""
    T, n = X.shape
    rank, size = _dist.world()
    lo, hi = _dist.block(T, rank, size)
    cnt = get_engine().band_halfspace_counts(X[lo:hi]) if hi > lo else np.zeros(n, dtype=np.int64)
    cnt = np.asarray(cnt, dtype=np.int64)
    return cnt if size == 1 else _dist.allreduce(cnt)
