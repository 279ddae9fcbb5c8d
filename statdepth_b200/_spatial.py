"""Functional spatial depth on the B200 engine (csrc/spatial.cu, DESIGN.md K14): the L2 spatial depth of curves
(Chakraborty & Chaudhuri 2014; depth.FSD in fda.usc).

A curve is the vector of its F = T d values in (t, c) order, compared by the plain Euclidean norm over all F values
(a uniform time weight would cancel inside u, so none is applied; channels are used as given).  With u(v) = v / ||v||
and u(0) = 0:

    SD(x_q) = 1 - || sum_{j : x_j != x_q} u(x_j - x_q) || / n

n counts x_q itself, and duplicates of x_q contribute 0.  Out of sample a new curve g is scored against the sample S
alone with the divisor n_S + 1: the depth FunctionalSpatialDepth(S + [g]) gives g, bit for bit.  The engine returns
r = ||sum u||; the host forms 1 - r / n_pop.

Sharding under `enable_distributed()`: every rank holds the whole sample and scores its block of the queries
(`_dist.query_sharded`); each query's sums run in an order fixed by the indices alone, so the depths equal one process
bit for bit.
"""
from typing import List

import numpy as np
import pandas as pd

from . import _dist
from ._engine import device_rows, get_engine
from ._functional import _positions
from ._reference import _curve_values

__all__ = ['_spatial_curves', '_functional_spatial', '_functional_spatial_of', '_SpatialReference']


def _rows(X, F):
    """The curves of (X [T, n], None) or (None, F [N, T, d]) as rows [n, T d] (a view where the memory allows)."""
    return X.T if X is not None else F.reshape(F.shape[0], -1)


def _spatial_curves(data: List[pd.DataFrame], frames=None):
    """(X, F) of data checked as FunctionalProjectionDepth checks curves; univariate data needs at least one curve."""
    X, F = _curve_values(data, frames=frames)
    if X is not None and X.shape[1] == 0:
        raise ValueError('No data passed.')
    return X, F


def _functional_spatial(data: List[pd.DataFrame], to_compute=None) -> pd.Series:
    """[df] (T x n, curves are columns; to_compute = column labels) or N DataFrames of T x d (one curve each;
    to_compute = list positions)."""
    X, F = _spatial_curves(data)
    A = _rows(X, F)
    n = A.shape[0]
    labels = (data[0].columns if X is not None else pd.RangeIndex(n)) if to_compute is None else to_compute
    axis = data[0].columns if X is not None else pd.RangeIndex(n)
    q = _positions(labels, axis, 'to_compute')
    r = _dist.query_sharded(lambda qb: get_engine().spatial_norms(A, qb), q, np.float64)
    index = list(labels) if X is None else labels
    return pd.Series(index=index, data=1.0 - np.asarray(r, dtype=np.float64) / n)


def _functional_spatial_of(data: List[pd.DataFrame], sample: List[pd.DataFrame]) -> pd.Series:
    """Depth of the new curves data against sample, each as if appended alone to it (one-shot, host buffers)."""
    XS, FS = _spatial_curves(sample)
    X, F = _checked_new_curves(data, XS, FS)
    S, Y = _rows(XS, FS), _rows(X, F)
    r = _dist.query_sharded(lambda qb: get_engine().spatial_norms_of(S, Y[qb]), np.arange(Y.shape[0]), np.float64)
    index = data[0].columns if X is not None else list(range(len(data)))
    return pd.Series(index=index, data=1.0 - np.asarray(r, dtype=np.float64) / (S.shape[0] + 1))


def _checked_new_curves(data, XS, FS):
    """(X, F) of the new curves, in the sample's form (univariate or frames), with its T (and d)."""
    X, F = _curve_values(data, frames=FS is not None)
    T = XS.shape[0] if XS is not None else FS.shape[1]
    if (X.shape[0] if X is not None else F.shape[1]) != T:
        raise ValueError('data and sample must have the same number of time points.')
    if F is not None and F.shape[2] != FS.shape[2]:
        raise ValueError('data and sample must have the same number of channels.')
    return X, F


class _SpatialReference:
    """A sample of curves kept for spatial depth: n_S x F doubles in a torch tensor on the engine's device for as long
    as the reference lives (a host array for a test double without `_dev` methods).  Every rank holds all of it."""

    def __init__(self, X=None, F=None):
        A = _rows(X, F)
        self.nS, self.F = A.shape
        self.eng = get_engine()
        self.on_device = hasattr(self.eng, 'spatial_norms_of_dev')
        if not self.on_device:
            self.sample = np.ascontiguousarray(A, dtype=np.float64)
            return
        import torch
        self.torch = torch
        _, self.sample = device_rows(self.eng, A)

    def _norms(self, Y):
        """r of the new curves Y [m, F] (rows) against the sample."""
        if not self.on_device:
            return self.eng.spatial_norms_of(self.sample, Y)
        torch = self.torch
        stream, dY = device_rows(self.eng, Y)
        with torch.cuda.stream(stream):
            out = torch.empty(Y.shape[0], dtype=torch.float64, device=dY.device)
            self.eng.spatial_norms_of_dev(self.sample.data_ptr(), self.nS, dY.data_ptr(), Y.shape[0], self.F,
                                          out.data_ptr())
            return out.cpu().numpy()

    def depths(self, Y: np.ndarray) -> np.ndarray:
        """Depth of every new curve: the columns of Y [T, nY] (univariate), else Y [nY, T, d]; each equals
        FunctionalSpatialDepth of the sample with that curve appended, bit for bit."""
        A = Y.T if Y.ndim == 2 else Y.reshape(Y.shape[0], -1)
        if A.shape[1] != self.F:
            raise ValueError('data and sample must have the same number of values per curve.')
        if A.shape[0] == 0:
            return np.zeros(0, dtype=np.float64)
        r = _dist.query_sharded(lambda qb: self._norms(A[qb]), np.arange(A.shape[0]), np.float64)
        return 1.0 - np.asarray(r, dtype=np.float64) / (self.nS + 1)

    def close(self) -> None:
        self.sample = None
