"""Kernelized functional spatial depth on the B200 engine (csrc/kfsd.cu, DESIGN.md K16): KFSD of Sguera, Galeano &
Lillo (2014), spatial depth after the feature map phi of a Gaussian kernel, which makes it local.

A curve is the vector of its F = T d values in (t, c) order, compared by the plain Euclidean norm, as in K14 and K15.
With k(x, y) = exp(-||x - y||^2 / sigma^2) and e = 1 - k (formed as -expm1, accurate for close curves):

    KFSD(x_q) = 1 - r_q / n,   r_q^2 = sum_{i, j in J_q} (e_qi + e_qj - e_ij) / (2 sqrt(e_qi e_qj))

J_q holds the curves with e_qj > 0, so x_q itself and its duplicates contribute 0, and n counts x_q.  r_q is the norm
of the sum of the feature-space unit vectors (phi(x_q) - phi(x_j)) / ||phi(x_q) - phi(x_j)||.  The engine returns r.
sigma is given, or np.quantile of the n (n - 1) / 2 pair distances at quantile (default 0.15), selected exactly as
for h-modal depth (_modal._selected_bandwidth): the same sample gives FunctionalModalDepth's bandwidth bits.  Out of
sample a new curve g is scored against the sample S with S's sigma and the divisor n_S + 1:
FunctionalKernelSpatialDepth(S + [g], bandwidth=sigma) gives g the same bits.

The engine keeps the sample's n x n matrix of e on the GPU, so n (n_S out of sample) is capped at KFSD_N_MAX.

Sharding under `enable_distributed()`: every rank selects sigma and builds E from the whole sample (the same bits as
one process) and scores its block of the queries (`_dist.query_sharded`).
"""
from typing import List

import numpy as np
import pandas as pd

from . import _dist
from ._engine import get_engine, resident
from ._functional import _positions
from ._modal import DEFAULT_QUANTILE, _checked_bandwidth, _selected_bandwidth
from ._spatial import _checked_new_curves, _rows, _spatial_curves

__all__ = ['KFSD_N_MAX', '_functional_kfsd', '_functional_kfsd_of', '_KfsdReference']

KFSD_N_MAX = 32768  # SD_KFSD_N_MAX (include/statdepth_b200.h): E holds n^2 doubles, 8 GiB at the cap


def _check_size(n: int, what: str) -> None:
    if n > KFSD_N_MAX:
        raise ValueError('kernelized spatial depth keeps the n x n kernel matrix on the GPU: %s has %d curves, at most '
                         '%d are supported' % (what, n, KFSD_N_MAX))


def _functional_kfsd(data: List[pd.DataFrame], to_compute=None, quantile=DEFAULT_QUANTILE,
                     bandwidth=None) -> pd.Series:
    """[df] (T x n, curves are columns; to_compute = column labels) or N DataFrames of T x d (one curve each;
    to_compute = list positions)."""
    h = _checked_bandwidth(quantile, bandwidth)
    X, F = _spatial_curves(data)
    A = _rows(X, F)
    n = A.shape[0]
    _check_size(n, 'the data')
    labels = (data[0].columns if X is not None else pd.RangeIndex(n)) if to_compute is None else to_compute
    axis = data[0].columns if X is not None else pd.RangeIndex(n)
    q = _positions(labels, axis, 'to_compute')
    eng = get_engine()
    R = resident(eng, A)  # one upload for the selection and the depth
    if h is None:
        h = _selected_bandwidth(eng, R, n, quantile)
    c = -1.0 / (h * h)
    r = _dist.query_sharded(lambda qb: eng.kfsd_norms(R, c, qb), q, np.float64)
    index = list(labels) if X is None else labels
    return pd.Series(index=index, data=1.0 - np.asarray(r, dtype=np.float64) / n)


def _functional_kfsd_of(data: List[pd.DataFrame], sample: List[pd.DataFrame], quantile=DEFAULT_QUANTILE,
                        bandwidth=None) -> pd.Series:
    """Depth of the new curves data against sample, each as if appended alone to it, with sample's bandwidth."""
    h = _checked_bandwidth(quantile, bandwidth)
    XS, FS = _spatial_curves(sample)
    X, F = _checked_new_curves(data, XS, FS)
    ref = _KfsdReference(X=XS, F=FS, quantile=quantile, bandwidth=h)
    try:
        depth = ref.depths(X if X is not None else F)
    finally:
        ref.close()
    index = data[0].columns if X is not None else list(range(len(data)))
    return pd.Series(index=index, data=depth)


class _KfsdReference:
    """A sample of curves kept for KFSD: n_S x F doubles uploaded once to the engine's device, its bandwidth, selected
    once at construction unless given, and its n_S x n_S matrix E of 1 - k, all kept for as long as the reference lives
    (E is 3.2 GB at n_S = 20 000).  Every rank holds all of it."""

    def __init__(self, X=None, F=None, quantile=DEFAULT_QUANTILE, bandwidth=None):
        h = _checked_bandwidth(quantile, bandwidth)
        A = _rows(X, F)
        self.nS, self.F = A.shape
        _check_size(self.nS, 'the sample')
        self.eng = get_engine()
        self.sample = resident(self.eng, A)
        self.bandwidth = h if h is not None else _selected_bandwidth(self.eng, self.sample, self.nS, quantile)
        self.c = -1.0 / (self.bandwidth * self.bandwidth)
        self.E = self.eng.kfsd_gram(self.sample, self.c)

    def depths(self, Y: np.ndarray) -> np.ndarray:
        """Depth of every new curve: the columns of Y [T, nY] (univariate), else Y [nY, T, d]; each equals
        FunctionalKernelSpatialDepth of the sample with that curve appended and bandwidth=self.bandwidth, bit for
        bit."""
        A = Y.T if Y.ndim == 2 else Y.reshape(Y.shape[0], -1)
        if A.shape[1] != self.F:
            raise ValueError('data and sample must have the same number of values per curve.')
        if A.shape[0] == 0:
            return np.zeros(0, dtype=np.float64)
        r = _dist.query_sharded(lambda qb: self.eng.kfsd_norms_of(self.sample, self.E, A[qb], self.c),
                                np.arange(A.shape[0]), np.float64)
        return 1.0 - np.asarray(r, dtype=np.float64) / (self.nS + 1)

    def close(self) -> None:
        self.sample = None
        self.E = None
