"""Random projection depths on the B200 engine (csrc/projection.cu, DESIGN.md K12): random Tukey depth
(Cuesta-Albertos & Nieto-Reyes 2008) and projection depth (Zuo & Serfling 2000) of point clouds and curves in any
dimension.

Every time point t and direction u give the projections y = u . x of the N values at t.  Random Tukey depth takes
h = N - max(b, a) per projection (b / a the other projections strictly below / above) and sums min_u h over t: an
exact int64 numerator R, depth R / (T N).  Projection depth takes O = max_u |y - med| / MAD (med and the unscaled
MAD of the projected row) and 1 / (1 + O), averaged over t for curves.

Directions: `directions=None` draws 1000, an int K draws K, both as
`np.random.default_rng(seed).standard_normal((K, d))` with every row divided by its `np.linalg.norm`; an array
[K, d] is used exactly as given.  Univariate curves have the single direction 1.0 (y = x).

Sharding under `enable_distributed()`: point clouds split the directions and all-reduce the MIN of the numerators
(Tukey) or the MAX of O (projection); curves split the time rows and all-reduce the SUM of the numerators (Tukey) or
all-gather the O rows (projection).  A rank without directions or rows contributes the identity.  Both are exact,
so the depths equal one process bit for bit.
"""
from typing import List

import numpy as np
import pandas as pd

from . import _dist
from ._engine import get_engine
from ._functional import _positions, _values
from ._halfspace import _functional_halfspace

__all__ = ['_pointcloud_projection', '_functional_projection', 'draw_directions', 'DEFAULT_DIRECTIONS']

DEFAULT_DIRECTIONS = 1000
KINDS = ('projection', 'tukey')


def draw_directions(d: int, directions=None, seed=0) -> np.ndarray:
    """The directions U [K, d] a call with these arguments uses (see the module docstring)."""
    if directions is None or (isinstance(directions, (int, np.integer)) and not isinstance(directions, bool)):
        K = DEFAULT_DIRECTIONS if directions is None else int(directions)
        if K < 1:
            raise ValueError('directions must be at least 1 (got %d)' % K)
        U = np.random.default_rng(seed).standard_normal((K, d))
        return np.stack([u / np.linalg.norm(u) for u in U])
    U = np.array(directions, dtype=np.float64)
    if U.ndim != 2 or U.shape[0] < 1 or U.shape[1] != d:
        raise ValueError('directions must be an int or an array of shape (K, %d), K >= 1 (got shape %s)'
                         % (d, U.shape))
    if not np.isfinite(U).all():
        raise ValueError('directions must be finite')
    if not (U != 0).any(axis=1).all():
        raise ValueError('every direction must be non-zero')
    return np.ascontiguousarray(U)


def _check_kind(kind):
    if kind not in KINDS:
        raise ValueError("kind must be one of %s (got %r)" % (KINDS, kind))


def _pointcloud_projection(data: pd.DataFrame, kind='projection', directions=None, seed=0,
                           to_compute=None) -> pd.Series:
    """Projection or random Tukey depth of the rows of the n x d cloud data, indexed by to_compute (all rows,
    data.index, when None)."""
    _check_kind(kind)
    if not isinstance(data, pd.DataFrame):
        raise ValueError('data must be a DataFrame (n points x d columns).')
    n, d = data.shape
    if n == 0 or d == 0:
        raise ValueError('No data passed.')
    U = draw_directions(d, directions, seed)
    if to_compute is None:
        to_compute = data.index
    q = _positions(to_compute, data.index, 'to_compute')
    F = np.ascontiguousarray(_values(data))[:, None, :]
    rank, size = _dist.world()
    lo, hi = _dist.block(len(U), rank, size)
    eng = get_engine() if hi > lo else None
    if kind == 'tukey':
        cnt = eng.projection_tukey_counts(F, U[lo:hi]) if hi > lo else np.full(n, n, dtype=np.int64)
        cnt = np.asarray(cnt, dtype=np.int64)
        if size > 1:
            cnt = _dist.allreduce(cnt, 'min')
        depth = cnt.astype(np.float64) / n
    else:
        o = eng.projection_outlyingness(F, U[lo:hi])[0] if hi > lo else np.zeros(n)
        o = np.asarray(o, dtype=np.float64)
        if size > 1:
            o = _dist.allreduce(o, 'max')
        depth = 1.0 / (1.0 + o)
    return pd.Series(index=to_compute, data=depth[q])


def _functional_projection(data: List[pd.DataFrame], kind='projection', directions=None, seed=0,
                           to_compute=None) -> pd.Series:
    """[df] (T x n, curves are columns; to_compute = column labels) or N DataFrames of T x d (one curve each;
    to_compute = list positions)."""
    _check_kind(kind)
    if not isinstance(data, list):
        raise ValueError('data must be passed as a list.')
    if len(data) == 0:
        raise ValueError('No data passed.')
    if len(data) == 1:
        if directions is not None:
            raise ValueError('univariate curves have the single direction 1.0: directions must be None')
        if kind == 'tukey':
            return _functional_halfspace(data, to_compute)
        df = data[0]
        T, n = df.shape
        if T == 0 or n == 0:
            raise ValueError('No data passed.')
        cols = df.columns if to_compute is None else to_compute
        q = None if to_compute is None else _positions(to_compute, df.columns, 'to_compute')
        X = _values(df)
        depth = _depth_from_rows(T, n, lambda lo, hi: get_engine().band_outlyingness(X[lo:hi]))
        return pd.Series(index=cols, data=depth if q is None else depth[q])
    if len({df.shape[1] for df in data}) > 1:
        raise ValueError('every curve must have the same number of channels.')
    if len({df.shape[0] for df in data}) > 1:
        raise ValueError('every curve must have the same number of time points.')
    N, (T, d) = len(data), data[0].shape
    if T == 0 or d == 0:
        raise ValueError('No data passed.')
    U = draw_directions(d, directions, seed)
    f = list(range(N)) if to_compute is None else to_compute
    q = _positions(f, pd.RangeIndex(N), 'to_compute')
    F = np.stack([_values(df) for df in data])
    rank, size = _dist.world()
    if kind == 'tukey':
        lo, hi = _dist.block(T, rank, size)
        cnt = (get_engine().projection_tukey_counts(np.ascontiguousarray(F[:, lo:hi]), U) if hi > lo
               else np.zeros(N, dtype=np.int64))
        cnt = np.asarray(cnt, dtype=np.int64)
        if size > 1:
            cnt = _dist.allreduce(cnt, 'sum')
        depth = cnt.astype(np.float64) / (T * N)
    else:
        depth = _depth_from_rows(T, N, lambda lo, hi: get_engine().projection_outlyingness(
            np.ascontiguousarray(F[:, lo:hi]), U))
    return pd.Series(index=f, data=depth[q])


def _depth_from_rows(T, n, outlyingness):
    """Projection depth of n curves from O [T, n]: this rank's block of time rows, all-gathered across ranks."""
    rank, size = _dist.world()
    lo, hi = _dist.block(T, rank, size)
    o = np.asarray(outlyingness(lo, hi), dtype=np.float64) if hi > lo else np.zeros((0, n))
    if size > 1:
        o = _dist.allgather_blocks(o, T)
    # C order: np.sum then adds the rows in order (its pairwise summation along a contiguous axis would differ)
    return np.sum(1.0 / (1.0 + np.ascontiguousarray(o)), axis=0) / T
